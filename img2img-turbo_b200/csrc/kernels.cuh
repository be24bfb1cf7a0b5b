// HBM-bound kernels of the path: GroupNorm(+SiLU), LayerNorm, softmax, layout / latent elementwise ops,
// and the load-time weight preparation (LoRA fold, TwinConv blend, re-layout, time-embedding constants).
// All activations are NHWC with an explicit pixel stride `ld` (elements) so channel slices are addressable.
#pragma once
#include "common.cuh"

namespace i2it {

// =============================================================================================
// GroupNorm (+SiLU)   — replaces ATen group_norm + silu at every norm1/norm2/conv_norm_out/
// Transformer2DModel.norm/attn.group_norm under the reference's vae.encode/unet/vae.decode calls
// (/root/reference/src/pix2pix_turbo.py:198-203).  Two launches: statistics (from the producing GEMM's epilogue partials, or
// one pass over the tensor; deterministic; the last block finalises in double) and apply.
// =============================================================================================
template <typename T>
__global__ void gn_stats_kernel(const T* __restrict__ x, long long img_stride, int ld, int C, int HW, int cg,
                                int pix_per_cta, float* __restrict__ partial /*[N][chunks][32][2]*/, int* __restrict__ counter,
                                double inv_count, float eps, float* __restrict__ stats /*[N][32] (mean, rstd)*/) {
  extern __shared__ float s_acc[];   // [rows][2][C]: per-row partials, reduced in a fixed order (bit-reproducible)
  const int vecs = C >> 3;
  const int vx = threadIdx.x % vecs, vy = threadIdx.x / vecs, rows = blockDim.x / vecs;
  const int n = blockIdx.y, chunk = blockIdx.x;
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
  const int p0 = chunk * pix_per_cta, p1 = min(HW, p0 + pix_per_cta);
  const T* xb = x + n * img_stride + vx * 8;
  auto acc = [&](const uint4& u) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = Elem<T>::unpack(w[i]);
      s[2 * i] += f.x; q[2 * i] += f.x * f.x;
      s[2 * i + 1] += f.y; q[2 * i + 1] += f.y * f.y;
    }
  };
  int p = p0 + vy;
  for (; p + 3 * rows < p1; p += 4 * rows) {           // 4 independent 16-byte loads in flight per thread
    const uint4 u0 = ld_nc16(xb + static_cast<long long>(p) * ld);
    const uint4 u1 = ld_nc16(xb + static_cast<long long>(p + rows) * ld);
    const uint4 u2 = ld_nc16(xb + static_cast<long long>(p + 2 * rows) * ld);
    const uint4 u3 = ld_nc16(xb + static_cast<long long>(p + 3 * rows) * ld);
    acc(u0); acc(u1); acc(u2); acc(u3);
  }
  for (; p < p1; p += rows) acc(ld_nc16(xb + static_cast<long long>(p) * ld));
  float* mine = s_acc + static_cast<size_t>(vy) * 2 * C;
#pragma unroll
  for (int i = 0; i < 8; ++i) { mine[vx * 8 + i] = s[i]; mine[C + vx * 8 + i] = q[i]; }
  __syncthreads();
  if (threadIdx.x < 32) {
    const int g = threadIdx.x;
    float a = 0.f, b = 0.f;
    for (int r = 0; r < rows; ++r) {
      const float* row = s_acc + static_cast<size_t>(r) * 2 * C;
      for (int c = g * cg; c < (g + 1) * cg; ++c) { a += row[c]; b += row[C + c]; }
    }
    float* o = partial + ((static_cast<long long>(n) * gridDim.x + chunk) * 32 + g) * 2;
    o[0] = a; o[1] = b;
    __threadfence();                                   // the partial is visible before this block's ticket is drawn
  }
  // Last level in the same launch: the block that draws image n's last ticket sums the chunk partials in ascending chunk
  // order (so the result does not depend on WHICH block is last: bit-reproducible) and writes (mean, rstd); it re-arms the
  // counter for the next replay.  The atomic orders the blocks, it never carries data.
  __shared__ int s_last;
  __shared__ double2 s_red[32][33];
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(&counter[n], 1) == static_cast<int>(gridDim.x) - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const int chunks = gridDim.x, g = threadIdx.x & 31, cl = threadIdx.x >> 5, ncl = blockDim.x >> 5;
  if (cl < ncl) {                                        // whole warps only (blockDim need not be a multiple of 32)
    const float2* base = reinterpret_cast<const float2*>(partial) + static_cast<long long>(n) * chunks * 32 + g;
    double a = 0.0, b = 0.0;
    for (int c = cl; c < chunks; c += ncl) {
      const float2 v = __ldcg(base + static_cast<long long>(c) * 32);
      a += static_cast<double>(v.x); b += static_cast<double>(v.y);
    }
    s_red[cl][g] = make_double2(a, b);
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < ncl; ++i) { a += s_red[i][g].x; b += s_red[i][g].y; }
    const double mean = a * inv_count;
    double var = b * inv_count - mean * mean;
    if (var < 0.0) var = 0.0;
    reinterpret_cast<float2*>(stats)[n * 32 + g] = make_float2(static_cast<float>(mean), static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps))));
  }
  if (threadIdx.x == 0) counter[n] = 0;
}

// Reduction of the partials a producing GEMM's epilogue wrote (TapGemmParams::gn_part, [phases][images][slots][per_row] x
// (sum, sumsq)): block (chunk, n) sums its share of image n's slots with COALESCED loads (threads run along the per_row entries
// of a slot row), folds the `epg` entries of each group -> scratch[n][chunk][32] in double; the block that draws the image's last
// ticket then sums the chunks in ascending order and writes (mean, rstd).  Up to 64 chunks per image so that the 2 MB of partials
// of a 512x512x128 image are pulled by 64 CTAs, not 4.  Fixed summation order: reproducible; the atomic only orders blocks.
static __global__ void gn_part_reduce_kernel(const float* __restrict__ part, int phases, int images, int slots, int per_row,
                                             int epg, int e_lanes /* pow2, <= 256 */, double2* __restrict__ scratch,
                                             int* __restrict__ counter, double inv_count, float eps, float* __restrict__ stats) {
  __shared__ double2 red[256];
  __shared__ double2 ent[640];                      // per_row <= 1280 / 2
  __shared__ int s_last;
  const int n = blockIdx.y, c = blockIdx.x, nch = gridDim.x, t = threadIdx.x;
  const int s0 = static_cast<int>(static_cast<long long>(c) * slots / nch), s1 = static_cast<int>(static_cast<long long>(c + 1) * slots / nch);
  const int nsl = 256 / e_lanes, te = t % e_lanes, tsl = t / e_lanes;
  for (int e0 = 0; e0 < per_row; e0 += e_lanes) {
    const int e = e0 + te;
    double a = 0.0, b = 0.0;
    if (e < per_row) {
      for (int ph = 0; ph < phases; ++ph) {
        const float2* base = reinterpret_cast<const float2*>(part) + (static_cast<long long>(ph) * images + n) * slots * per_row + e;
        int sl = s0 + tsl;
        for (; sl + 3 * nsl < s1; sl += 4 * nsl) {           // 4 independent loads in flight
          const float2 v0 = base[static_cast<long long>(sl) * per_row], v1 = base[static_cast<long long>(sl + nsl) * per_row];
          const float2 v2 = base[static_cast<long long>(sl + 2 * nsl) * per_row], v3 = base[static_cast<long long>(sl + 3 * nsl) * per_row];
          a += static_cast<double>(v0.x); b += static_cast<double>(v0.y);
          a += static_cast<double>(v1.x); b += static_cast<double>(v1.y);
          a += static_cast<double>(v2.x); b += static_cast<double>(v2.y);
          a += static_cast<double>(v3.x); b += static_cast<double>(v3.y);
        }
        for (; sl < s1; sl += nsl) {
          const float2 v = base[static_cast<long long>(sl) * per_row];
          a += static_cast<double>(v.x); b += static_cast<double>(v.y);
        }
      }
    }
    red[t] = make_double2(a, b);
    __syncthreads();
    if (tsl == 0 && e < per_row) {
      double2 acc = red[te];
      for (int k = 1; k < nsl; ++k) { acc.x += red[k * e_lanes + te].x; acc.y += red[k * e_lanes + te].y; }
      ent[e] = acc;
    }
    __syncthreads();
  }
  if (t < 32) {
    double2 acc = make_double2(0.0, 0.0);
    for (int k = 0; k < epg; ++k) { acc.x += ent[t * epg + k].x; acc.y += ent[t * epg + k].y; }
    scratch[(static_cast<long long>(n) * nch + c) * 32 + t] = acc;
    __threadfence();
  }
  __syncthreads();
  if (t == 0) s_last = (atomicAdd(&counter[n], 1) == nch - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  // last block of image n: thread (k-lane, g) sums chunks k-lane, k-lane + 8, ... ; lanes combined in a fixed order
  const int g = t & 31, kl = t >> 5;
  double a = 0.0, b = 0.0;
  for (int k = kl; k < nch; k += 8) {
    const double2 v = __ldcg(scratch + (static_cast<long long>(n) * nch + k) * 32 + g);
    a += v.x; b += v.y;
  }
  red[t] = make_double2(a, b);
  __syncthreads();
  if (t < 32) {
    a = 0.0; b = 0.0;
    for (int i = 0; i < 8; ++i) { a += red[i * 32 + t].x; b += red[i * 32 + t].y; }
    const double mean = a * inv_count;
    double var = b * inv_count - mean * mean;
    if (var < 0.0) var = 0.0;
    reinterpret_cast<float2*>(stats)[n * 32 + t] = make_float2(static_cast<float>(mean), static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps))));
  }
  if (t == 0) counter[n] = 0;
}

template <typename T>
__global__ void gn_apply_kernel(const T* __restrict__ x, long long ximg, int ldx, T* __restrict__ y, long long yimg,
                                int ldy, int C, int HW, int cg, int pix_per_cta, const float* __restrict__ stats,
                                const float* __restrict__ gamma, const float* __restrict__ beta, int silu) {
  const int vecs = C >> 3;
  const int vx = threadIdx.x % vecs, vy = threadIdx.x / vecs, rows = blockDim.x / vecs;
  const int n = blockIdx.y;
  if (vy >= rows) return;
  float sc[8], sh[8];
  int gprev = -1;
  float mean = 0.f, rstd = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = vx * 8 + i, g = c / cg;
    if (g != gprev) {                 // (mean, rstd) were finalised by the statistics launch (last-block reduction)
      gprev = g;
      const float2 mr = reinterpret_cast<const float2*>(stats)[n * 32 + g];
      mean = mr.x; rstd = mr.y;
    }
    sc[i] = rstd * gamma[c];
    sh[i] = beta[c] - mean * sc[i];
  }
  const int p0 = blockIdx.x * pix_per_cta, p1 = min(HW, p0 + pix_per_cta);
  const T* xb = x + n * ximg + vx * 8;
  T* yb = y + n * yimg + vx * 8;
  auto xf = [&](const uint4& u) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    uint32_t o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = Elem<T>::unpack(w[i]);
      float a = f.x * sc[2 * i] + sh[2 * i], b = f.y * sc[2 * i + 1] + sh[2 * i + 1];
      if (silu) { a = silu_f(a); b = silu_f(b); }
      o[i] = Elem<T>::pack(a, b);
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
  };
  int p = p0 + vy;
  for (; p + 3 * rows < p1; p += 4 * rows) {
    const uint4 u0 = ld_nc16(xb + static_cast<long long>(p) * ldx);
    const uint4 u1 = ld_nc16(xb + static_cast<long long>(p + rows) * ldx);
    const uint4 u2 = ld_nc16(xb + static_cast<long long>(p + 2 * rows) * ldx);
    const uint4 u3 = ld_nc16(xb + static_cast<long long>(p + 3 * rows) * ldx);
    st16(yb + static_cast<long long>(p) * ldy, xf(u0));
    st16(yb + static_cast<long long>(p + rows) * ldy, xf(u1));
    st16(yb + static_cast<long long>(p + 2 * rows) * ldy, xf(u2));
    st16(yb + static_cast<long long>(p + 3 * rows) * ldy, xf(u3));
  }
  for (; p < p1; p += rows) st16(yb + static_cast<long long>(p) * ldy, xf(ld_nc16(xb + static_cast<long long>(p) * ldx)));
}

// =============================================================================================
// LayerNorm over the channel dim of token rows (BasicTransformerBlock.norm1/2/3), one warp per row.
// =============================================================================================
template <typename T>
__global__ void layernorm_kernel(const T* __restrict__ x, int ldx, T* __restrict__ y, int ldy, int rows, int C,
                                 const float* __restrict__ gamma, const float* __restrict__ beta, float eps) {
  constexpr int MAXV = 5;   // C <= 1280
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const int vecs = C >> 3;
  float v[MAXV][8];
  float sum = 0.f;
  const T* xr = x + static_cast<long long>(warp) * ldx;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int vi = lane + 32 * k;
    if (vi < vecs) {
      const uint4 u = ld_nc16(xr + vi * 8);
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = Elem<T>::unpack(w[i]);
        v[k][2 * i] = f.x; v[k][2 * i + 1] = f.y;
        sum += f.x + f.y;
      }
    }
  }
  const float mean = warp_sum(sum) / C;
  float sq = 0.f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    if (lane + 32 * k < vecs) {
#pragma unroll
      for (int i = 0; i < 8; ++i) { const float d = v[k][i] - mean; sq += d * d; }
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / C + eps);
  T* yr = y + static_cast<long long>(warp) * ldy;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int vi = lane + 32 * k;
    if (vi < vecs) {
      uint32_t o[4];
      const float4 g0 = *reinterpret_cast<const float4*>(gamma + vi * 8), g1 = *reinterpret_cast<const float4*>(gamma + vi * 8 + 4);
      const float4 b0 = *reinterpret_cast<const float4*>(beta + vi * 8), b1 = *reinterpret_cast<const float4*>(beta + vi * 8 + 4);
      const float gm[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float bt[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        o[i] = Elem<T>::pack((v[k][2 * i] - mean) * rstd * gm[2 * i] + bt[2 * i],
                             (v[k][2 * i + 1] - mean) * rstd * gm[2 * i + 1] + bt[2 * i + 1]);
      }
      st16(yr + vi * 8, make_uint4(o[0], o[1], o[2], o[3]));
    }
  }
}

// =============================================================================================
// Row softmax: fp32 logits (already scaled) -> probabilities in the activation dtype.
// TPR threads cooperate on one row (32 or 128); up to 32 values per thread live in registers.
// =============================================================================================
template <typename T, int TPR>
__global__ void softmax_kernel(const float* __restrict__ s, long long lds, T* __restrict__ pr, long long ldp,
                               long long rows, int nk, int nk_pad) {
  constexpr int RPB = 128 / TPR;
  const long long row = static_cast<long long>(blockIdx.x) * RPB + threadIdx.x / TPR;
  const int tr = threadIdx.x % TPR;
  __shared__ float red[4];
  const bool ok = row < rows;
  const float* sr = s + (ok ? row : 0) * lds;
  float v[32];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = tr + i * TPR;
    v[i] = (ok && c < nk) ? sr[c] : -INFINITY;
    m = fmaxf(m, v[i]);
  }
  m = warp_max(m);
  if (TPR == 128) {
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
    __syncthreads();
  }
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = tr + i * TPR;
    v[i] = (c < nk) ? __expf(v[i] - m) : 0.f;
    sum += v[i];
  }
  sum = warp_sum(sum);
  if (TPR == 128) {
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    sum = red[0] + red[1] + red[2] + red[3];
  }
  if (!ok) return;
  const float inv = 1.0f / sum;
  T* o = pr + row * ldp;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = tr + i * TPR;
    if (c < nk_pad) o[c] = Elem<T>::from_f(c < nk ? v[i] * inv : 0.f);
  }
}

// Row softmax for rows longer than 4096 logits (VAE attention of images larger than 512x512): one CTA of 256 threads per row,
// three strided passes over the fp32 logits (max, sum, write) — the logits of one row (<= a few tens of KB) stay in L1/L2.
template <typename T>
__global__ void softmax_long_kernel(const float* __restrict__ s, long long lds, T* __restrict__ pr, long long ldp, int nk, int nk_pad) {
  __shared__ float red[8];
  const long long row = blockIdx.x;
  const float* sr = s + row * lds;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float m = -INFINITY;
  for (int c = threadIdx.x; c < nk; c += 256) m = fmaxf(m, sr[c]);
  m = warp_max(m);
  if (lane == 0) red[w] = m;
  __syncthreads();
  m = red[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
  __syncthreads();
  float sum = 0.f;
  for (int c = threadIdx.x; c < nk; c += 256) sum += __expf(sr[c] - m);
  sum = warp_sum(sum);
  if (lane == 0) red[w] = sum;
  __syncthreads();
  sum = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) sum += red[i];          // fixed order: reproducible
  const float inv = 1.0f / sum;
  T* o = pr + row * ldp;
  for (int c = threadIdx.x; c < nk_pad; c += 256) o[c] = Elem<T>::from_f(c < nk ? __expf(sr[c] - m) * inv : 0.f);
}

// =============================================================================================
// CLIP text embeddings: out[b, t, :] = token_embedding[ids[b, t]] + position_embedding[t]   (fp32 add, one rounding)
// (transformers models/clip/modeling_clip.py CLIPTextEmbeddings.forward; reference call /root/reference/src/pix2pix_turbo.py:190-196)
// =============================================================================================
template <typename T>
__global__ void clip_embed_kernel(const int* __restrict__ ids, const float* __restrict__ tok, const float* __restrict__ pos,
                                  T* __restrict__ out, int C, int ntok, int vocab, long long total /* rows * C/8 */) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int vecs = C >> 3;
  const long long r = i / vecs;
  const int v = static_cast<int>(i % vecs);
  const int t = static_cast<int>(r % ntok);
  int id = ids[r];
  id = min(max(id, 0), vocab - 1);
  const float4* a = reinterpret_cast<const float4*>(tok + static_cast<long long>(id) * C + v * 8);
  const float4* b = reinterpret_cast<const float4*>(pos + static_cast<long long>(t) * C + v * 8);
  const float4 a0 = a[0], a1 = a[1], b0 = b[0], b1 = b[1];
  st16(out + r * C + v * 8, make_uint4(Elem<T>::pack(a0.x + b0.x, a0.y + b0.y), Elem<T>::pack(a0.z + b0.z, a0.w + b0.w),
                                       Elem<T>::pack(a1.x + b1.x, a1.y + b1.y), Elem<T>::pack(a1.z + b1.z, a1.w + b1.w)));
}

// =============================================================================================
// boundary + latent elementwise kernels
// =============================================================================================
// NCHW [B,3,H,W] (act dtype) -> NHWC8 (channels 3..7 zero): the 3-channel boundary of vae.encode.
template <typename T>
__global__ void pack_input_kernel(const T* __restrict__ x, T* __restrict__ y, int C, long long HW, long long total) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // over B*HW pixels
  if (i >= total) return;
  const long long n = i / HW, p = i % HW;
  uint32_t o[4] = {0, 0, 0, 0};
  float c[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) c[k] = (k < C) ? Elem<T>::to_f(x[(n * C + k) * HW + p]) : 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) o[k] = Elem<T>::pack(c[2 * k], c[2 * k + 1]);
  st16(y + i * 8, make_uint4(o[0], o[1], o[2], o[3]));
}

// NCHW [B,3,H,W] -> im2col rows [B,H,W,32]: k = (ky*3+kx)*3 + c for the 3x3 pad-1 neighbourhood (27 values, 5 zeros).
// Turns encoder.conv_in (Cin=3: 16-byte TMA rows x 9 taps, TMA-request bound) into ONE K=32 GEMM tap with 64-byte rows.
template <typename T>
__global__ void pack_input_im2col_kernel(const T* __restrict__ x, T* __restrict__ y, int H, int W, long long total) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // over B*H*W pixels
  if (i >= total) return;
  const long long HW = static_cast<long long>(H) * W;
  const long long n = i / HW;
  const int p = static_cast<int>(i % HW), py = p / W, px = p % W;
  float v[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) v[k] = 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int yy = py + ky - 1, xx = px + kx - 1;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
#pragma unroll
        for (int c = 0; c < 3; ++c) v[(ky * 3 + kx) * 3 + c] = Elem<T>::to_f(x[(n * 3 + c) * HW + static_cast<long long>(yy) * W + xx]);
      }
    }
#pragma unroll
  for (int g = 0; g < 4; ++g)
    st16(y + i * 32 + g * 8, make_uint4(Elem<T>::pack(v[8 * g], v[8 * g + 1]), Elem<T>::pack(v[8 * g + 2], v[8 * g + 3]),
                                        Elem<T>::pack(v[8 * g + 4], v[8 * g + 5]), Elem<T>::pack(v[8 * g + 6], v[8 * g + 7])));
}

// uint8 HWC boundary (SURVEY section 8f #3).  Input: what the reference CLIs do on the host before the forward —
//   mode 0  F.to_tensor(img)                      v = u8/255                      (/root/reference/src/inference_paired.py:50)
//   mode 1  ToTensor + Normalize([0.5],[0.5])     v = (u8/255 - 0.5)/0.5          (/root/reference/src/inference_unpaired.py:45-47)
//   mode 2  (F.to_tensor(img) < 0.5).float()      v = u8/255 < 0.5 ? 1 : 0        (/root/reference/src/inference_paired.py:56-57)
// in fp32 followed by the .half()/.to(dtype) rounding — fused with the im2col packing of encoder.conv_in.
__device__ __forceinline__ float u8_to_input(uint8_t q, int mode) {
  const float v = static_cast<float>(q) / 255.0f;
  if (mode == 1) return (v - 0.5f) / 0.5f;
  if (mode == 2) return v < 0.5f ? 1.0f : 0.0f;
  return v;
}
template <typename T>
__global__ void pack_input_im2col_u8_kernel(const uint8_t* __restrict__ x /*[B,H,W,3]*/, T* __restrict__ y, int H, int W,
                                            long long total, int mode) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // over B*H*W pixels
  if (i >= total) return;
  const long long HW = static_cast<long long>(H) * W;
  const long long n = i / HW;
  const int p = static_cast<int>(i % HW), py = p / W, px = p % W;
  float v[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) v[k] = 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int yy = py + ky - 1, xx = px + kx - 1;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
        const uint8_t* q = x + ((n * H + yy) * W + xx) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) v[(ky * 3 + kx) * 3 + c] = Elem<T>::to_f(Elem<T>::from_f(u8_to_input(q[c], mode)));
      }
    }
#pragma unroll
  for (int g = 0; g < 4; ++g)
    st16(y + i * 32 + g * 8, make_uint4(Elem<T>::pack(v[8 * g], v[8 * g + 1]), Elem<T>::pack(v[8 * g + 2], v[8 * g + 3]),
                                        Elem<T>::pack(v[8 * g + 4], v[8 * g + 5]), Elem<T>::pack(v[8 * g + 6], v[8 * g + 7])));
}
// Output: transforms.ToPILImage()(output_image[0].cpu() * 0.5 + 0.5)  (/root/reference/src/inference_paired.py:72,
// /root/reference/src/inference_unpaired.py:53): three ops in the activation dtype (x*0.5, +0.5, .mul(255)), each rounded, then
// .byte() (truncation).  NCHW [B,3,H,W] -> HWC uint8 [B,H,W,3].
template <typename T>
__global__ void nchw_to_u8hwc_kernel(const T* __restrict__ x, uint8_t* __restrict__ y, long long HW, long long total) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // over B*H*W pixels
  if (i >= total) return;
  const long long n = i / HW, p = i % HW;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float a = Elem<T>::to_f(Elem<T>::from_f(Elem<T>::to_f(x[(n * 3 + c) * HW + p]) * 0.5f));
    const float b = Elem<T>::to_f(Elem<T>::from_f(a + 0.5f));
    const float d = Elem<T>::to_f(Elem<T>::from_f(b * 255.0f));
    y[i * 3 + c] = static_cast<uint8_t>(fminf(fmaxf(d, 0.f), 255.f));
  }
}

// DiagonalGaussianDistribution.sample() * scaling_factor (+ the stochastic blend of
// /root/reference/src/pix2pix_turbo.py:210): moments NHWC (ld) -> latent NHWC8 (channels 4..7 zero).
template <typename T>
__global__ void latent_sample_kernel(const T* __restrict__ mom, int ldm, const T* __restrict__ eps_nchw,
                                     const T* __restrict__ noise_nchw, float r, float sf, T* __restrict__ z,
                                     long long HW, long long total) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long n = i / HW, p = i % HW;
  float o[8];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float mean = Elem<T>::to_f(mom[i * ldm + c]);
    const float logvar = fminf(fmaxf(Elem<T>::to_f(mom[i * ldm + 4 + c]), -30.f), 20.f);
    const float e = Elem<T>::to_f(eps_nchw[(n * 4 + c) * HW + p]);
    float v = (mean + expf(0.5f * logvar) * e) * sf;
    if (noise_nchw) {
      // reference rounds the encoded latent to the activation dtype before blending
      v = Elem<T>::to_f(Elem<T>::from_f(v)) * r + Elem<T>::to_f(noise_nchw[(n * 4 + c) * HW + p]) * (1.f - r);
    }
    o[c] = v;
  }
#pragma unroll
  for (int c = 4; c < 8; ++c) o[c] = 0.f;
  st16(z + i * 8, make_uint4(Elem<T>::pack(o[0], o[1]), Elem<T>::pack(o[2], o[3]), 0u, 0u));
}

// DDPMScheduler.step closed form at t=999 and the `/ scaling_factor` feeding vae.decode
// (/root/reference/src/pix2pix_turbo.py:200-203): x0 = (x - s1*eps_hat)/sa.
//   three_round == 0  Pix2Pix_Turbo: `timesteps` is a 1-D tensor, so alphas_cumprod[t] is a dimensioned fp32 tensor and the
//                     whole step is promoted to fp32, then rounded once by .to(model_pred.dtype)  (pix2pix_turbo.py:162,200-201)
//   three_round == 1  CycleGAN_Turbo: `timesteps[i]` is 0-dim, so alphas_cumprod[t] (moved to the GPU by make_1step_sched,
//                     /root/reference/src/model.py:10) is a 0-dim CUDA fp32 tensor: it does not promote the fp16/bf16 operands,
//                     torch casts it to the activation dtype and every op rounds: c1 = round(s1), c2 = round(sa);
//                     round(c1*e), round(x - .), round(. / c2) with fp32 op-math  (/root/reference/src/cyclegan_turbo.py:205).
//                     tests/test_gpu_boundary.py checks this bit for bit against the same torch expression on the GPU.
template <typename T>
__global__ void ddpm_step_kernel(const T* __restrict__ zin /*NHWC8*/, const T* __restrict__ pred, int ldp,
                                 float s1, float sa, float inv_sf, T* __restrict__ dec_in /*NHWC8*/,
                                 T* __restrict__ x0_nchw /*nullable*/, long long HW, long long total, int three_round) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long n = i / HW, p = i % HW;
  float o[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float x = Elem<T>::to_f(zin[i * 8 + c]), e = Elem<T>::to_f(pred[i * ldp + c]);
    T x0t;
    if (three_round) {
      const float c1 = Elem<T>::to_f(Elem<T>::from_f(s1)), c2 = Elem<T>::to_f(Elem<T>::from_f(sa));
      const float t1 = Elem<T>::to_f(Elem<T>::from_f(c1 * e));
      const float t2 = Elem<T>::to_f(Elem<T>::from_f(x - t1));
      x0t = Elem<T>::from_f(t2 / c2);
    } else {
      x0t = Elem<T>::from_f((x - s1 * e) / sa);                  // x_denoised.to(dtype)
    }
    if (x0_nchw) x0_nchw[(n * 4 + c) * HW + p] = x0t;
    o[c] = Elem<T>::to_f(x0t) * inv_sf;
  }
  st16(dec_in + i * 8, make_uint4(Elem<T>::pack(o[0], o[1]), Elem<T>::pack(o[2], o[3]), 0u, 0u));
}

// nearest upsample to (Ho, Wo), NHWC, 16-byte vectors.  Index rule of F.interpolate(mode="nearest"): src = min(floor(dst * in/out),
// in - 1) with the ratio in fp32 (exactly 2x when Ho = 2H).  diffusers Upsample2D passes an explicit output size when the latent
// is not a multiple of 8 (UNet2DConditionModel.forward: forward_upsample_size), e.g. 14 -> 27 for a 560x840 image.
template <typename T>
__global__ void upsample_nearest_kernel(const T* __restrict__ x, int ldx, T* __restrict__ y, int ldy, int H, int W, int Ho, int Wo,
                                        float sh, float sw, int C, long long total /* B*Ho*Wo*(C/8) */) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int vecs = C >> 3;
  const int v = static_cast<int>(i % vecs);
  long long p = i / vecs;
  const int ox = static_cast<int>(p % Wo); p /= Wo;
  const int oy = static_cast<int>(p % Ho);
  const long long n = p / Ho;
  const int sy = min(static_cast<int>(floorf(oy * sh)), H - 1), sx = min(static_cast<int>(floorf(ox * sw)), W - 1);
  const uint4 u = ld_nc16(x + ((n * H + sy) * W + sx) * ldx + v * 8);
  st16(y + ((n * Ho + oy) * Wo + ox) * ldy + v * 8, u);
}

// zero-padded copy [B,H,W,C] -> [B,H2,W2,C] (H2 >= H, W2 >= W): a stride-2 conv over an odd-sized map reads the 5-D parity view
// of an EVEN-sized tensor, and its right/bottom zero padding becomes real zeros
template <typename T>
__global__ void pad_copy_kernel(const T* __restrict__ x, int ldx, T* __restrict__ y, int H, int W, int H2, int W2, int C,
                                long long total /* B*H2*W2*(C/8) */) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int vecs = C >> 3;
  const int v = static_cast<int>(i % vecs);
  long long p = i / vecs;
  const int ox = static_cast<int>(p % W2); p /= W2;
  const int oy = static_cast<int>(p % H2);
  const long long n = p / H2;
  uint4 u = make_uint4(0u, 0u, 0u, 0u);
  if (oy < H && ox < W) u = ld_nc16(x + ((n * H + oy) * W + ox) * ldx + v * 8);
  st16(y + ((n * H2 + oy) * W2 + ox) * C + v * 8, u);
}

// split-K epilogue: out[r][c] = round( sum_s part[s][r][c] + bias[c] + res[r][c] ), partials summed in index order (reproducible)
template <typename T>
__global__ void splitk_reduce_kernel(const float* __restrict__ part, int S, long long split_stride, const float* __restrict__ bias,
                                     const T* __restrict__ res, int ldr, T* __restrict__ out, int ldo, int N, long long total /* rows*N/8 */) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int vecs = N >> 3;
  const long long r = i / vecs;
  const int c0 = static_cast<int>(i % vecs) * 8;
  float v[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = bias ? bias[c0 + k] : 0.f;
  for (int s = 0; s < S; ++s) {
    const float4* p4 = reinterpret_cast<const float4*>(part + s * split_stride + r * N + c0);
    const float4 a = p4[0], b = p4[1];
    v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w; v[4] += b.x; v[5] += b.y; v[6] += b.z; v[7] += b.w;
  }
  if (res) {
    const uint4 u = ld_nc16(res + r * ldr + c0);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float2 f = Elem<T>::unpack(w[k]); v[2 * k] += f.x; v[2 * k + 1] += f.y; }
  }
  st16(out + r * ldo + c0, make_uint4(Elem<T>::pack(v[0], v[1]), Elem<T>::pack(v[2], v[3]), Elem<T>::pack(v[4], v[5]), Elem<T>::pack(v[6], v[7])));
}

// strided 2-D copy of 16-byte vectors: rows x (C/8) vectors (torch.cat along channels)
template <typename T>
__global__ void copy2d_kernel(const T* __restrict__ x, int ldx, T* __restrict__ y, int ldy, int C, long long total) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int vecs = C >> 3;
  const long long r = i / vecs;
  const int v = static_cast<int>(i % vecs);
  st16(y + r * ldy + v * 8, ld_nc16(x + r * ldx + v * 8));
}

}  // namespace i2it
