// Canny edge map on the device, bit-exact with OpenCV's cv2.Canny(img, low, high) (apertureSize 3, L1 gradient) on 8-bit
// 3-channel images: the control image of the edge_to_image model (the reference's src/image_prep.py:6-12).
//
//   canny_tile_kernel    one CTA per 32x32 tile: Sobel (replicated border) on all 3 channels over the tile + 1-px ring, the
//                        channel with the largest |dx|+|dy| (first on a tie), fixed-point non-maximum suppression (zero
//                        magnitude outside the image), weak/strong classification, and a union-find over the tile's
//                        candidates in shared memory.  Writes class, the tile-local root as a global label, clears flags.
//   canny_merge_kernel   joins components across tile borders in global memory (atomicMin union, Playne & Hawick,
//                        IEEE TPDS 2018).  Invariant label[p] <= p: every find() walk terminates.
//   canny_mark_kernel    every candidate points its label straight at its root; strong ones set flag[root].
//   canny_out_kernel     255 for candidates whose root is flagged, else 0, three identical channels, 16-byte stores.
//
// The atomics only decide which pixel becomes a component's root (always its smallest index); the output is "does the
// component contain a strong pixel", so it is deterministic.  Hysteresis is exact for components of any length: there is
// no bounded number of propagation sweeps.  Workspace: label int32 + class u8 + flag u8 per pixel.
#pragma once
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace i2it {

constexpr int CANNY_TILE = 32;
constexpr int CANNY_THREADS = 256;

struct CannyWs {
  int* label;        // union-find parent (candidates only)
  uint8_t* cls;      // 0 none, 1 weak candidate, 2 strong candidate
  uint8_t* flag;     // 1 at roots of components that contain a strong pixel
};

inline size_t canny_align16(size_t b) { return (b + 15) & ~static_cast<size_t>(15); }
inline size_t canny_workspace_bytes(long long n) {
  return canny_align16(4 * static_cast<size_t>(n)) + 2 * canny_align16(static_cast<size_t>(n));
}
inline CannyWs canny_ws(void* base, long long n) {
  char* p = static_cast<char*>(base);
  CannyWs w;
  w.label = reinterpret_cast<int*>(p);
  w.cls = reinterpret_cast<uint8_t*>(p + canny_align16(4 * static_cast<size_t>(n)));
  w.flag = w.cls + canny_align16(static_cast<size_t>(n));
  return w;
}

// Root of x.  Parents only ever decrease and never exceed the child, so the walk ends; volatile reads see other threads'
// atomicMin updates (shared or global memory alike).
__device__ __forceinline__ int canny_find(const int* label, int x) {
  int l = *reinterpret_cast<const volatile int*>(label + x);
  while (l != x) {
    x = l;
    l = *reinterpret_cast<const volatile int*>(label + x);
  }
  return x;
}

// Join the sets of a and b: the larger root is hooked under the smaller one; retried when another thread moved it first.
__device__ __forceinline__ void canny_union(int* label, int a, int b) {
  bool done;
  do {
    a = canny_find(label, a);
    b = canny_find(label, b);
    if (a < b) {
      const int old = atomicMin(label + b, a);
      done = old == b;
      b = old;
    } else if (b < a) {
      const int old = atomicMin(label + a, b);
      done = old == a;
      a = old;
    } else {
      done = true;
    }
  } while (!done);
}

static __global__ void __launch_bounds__(CANNY_THREADS)
canny_tile_kernel(const uint8_t* __restrict__ x, int H, int W, int lo, int hi, CannyWs ws) {
  constexpr int T = CANNY_TILE, R = T + 2, I = T + 4;
  __shared__ uint8_t s_in[I * I * 3];   // input rows / cols tile0-2 .. tile0+T+1, clamped coordinates (replicated border)
  __shared__ int s_mag[R * R];          // magnitude over rows / cols tile0-1 .. tile0+T, 0 outside the image
  __shared__ short2 s_d[T * T];         // dx, dy of the selected channel at the tile's own pixels
  __shared__ int s_lab[T * T];
  __shared__ uint8_t s_cls[T * T];
  const int b = blockIdx.z, ty0 = blockIdx.y * T, tx0 = blockIdx.x * T;
  const long long img0 = static_cast<long long>(b) * H * W;
  const uint8_t* img = x + img0 * 3;

  for (int i = threadIdx.x; i < I * I; i += CANNY_THREADS) {
    const int r = i / I, c = i - r * I;
    const int gy = min(max(ty0 - 2 + r, 0), H - 1), gx = min(max(tx0 - 2 + c, 0), W - 1);
    const uint8_t* p = img + (static_cast<long long>(gy) * W + gx) * 3;
    s_in[i * 3 + 0] = p[0];
    s_in[i * 3 + 1] = p[1];
    s_in[i * 3 + 2] = p[2];
  }
  __syncthreads();

  for (int i = threadIdx.x; i < R * R; i += CANNY_THREADS) {
    const int r = i / R, c = i - r * R;
    const int gy = ty0 - 1 + r, gx = tx0 - 1 + c;
    int best = 0, bdx = 0, bdy = 0;
    if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
      const uint8_t* q = s_in + (r * I + c) * 3;   // top-left of the 3x3 window centred on (gy, gx)
      best = -1;
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
        auto at = [&](int dr, int dc) { return static_cast<int>(q[(dr * I + dc) * 3 + ch]); };
        const int dx = (at(0, 2) + 2 * at(1, 2) + at(2, 2)) - (at(0, 0) + 2 * at(1, 0) + at(2, 0));
        const int dy = (at(2, 0) + 2 * at(2, 1) + at(2, 2)) - (at(0, 0) + 2 * at(0, 1) + at(0, 2));
        const int m = abs(dx) + abs(dy);
        if (m > best) { best = m; bdx = dx; bdy = dy; }
      }
    }
    s_mag[i] = best;
    if (r >= 1 && r <= T && c >= 1 && c <= T) s_d[(r - 1) * T + (c - 1)] = make_short2(bdx, bdy);
  }
  __syncthreads();

  for (int i = threadIdx.x; i < T * T; i += CANNY_THREADS) {
    const int ly = i / T, lx = i % T;
    int cl = 0;
    if (ty0 + ly < H && tx0 + lx < W) {
      const int* mp = s_mag + (ly + 1) * R + lx + 1;
      const int m = *mp;
      if (m > lo) {
        const short2 d = s_d[i];
        const int ax = abs(d.x), ay = abs(d.y) << 15;   // |d| <= 1020: all products below fit in int32
        const int tg22 = ax * 13573, tg67 = tg22 + (ax << 16);
        bool keep;
        if (ay < tg22) {
          keep = m > mp[-1] && m >= mp[1];
        } else if (ay > tg67) {
          keep = m > mp[-R] && m >= mp[R];
        } else {
          const int s = (d.x ^ d.y) < 0 ? -1 : 1;
          keep = m > mp[-R - s] && m > mp[R + s];
        }
        if (keep) cl = m > hi ? 2 : 1;
      }
    }
    s_cls[i] = static_cast<uint8_t>(cl);
    s_lab[i] = i;
  }
  __syncthreads();

  // tile-local components: join every candidate with its candidate neighbours left, up-left, up, up-right
  for (int i = threadIdx.x; i < T * T; i += CANNY_THREADS) {
    if (!s_cls[i]) continue;
    const int ly = i / T, lx = i % T;
    if (lx > 0 && s_cls[i - 1]) canny_union(s_lab, i, i - 1);
    if (ly > 0) {
      if (lx > 0 && s_cls[i - T - 1]) canny_union(s_lab, i, i - T - 1);
      if (s_cls[i - T]) canny_union(s_lab, i, i - T);
      if (lx < T - 1 && s_cls[i - T + 1]) canny_union(s_lab, i, i - T + 1);
    }
  }
  __syncthreads();

  // local index order (row-major) is global index order inside a tile, so the root stays <= p globally as well
  for (int i = threadIdx.x; i < T * T; i += CANNY_THREADS) {
    const int ly = i / T, lx = i % T;
    if (ty0 + ly >= H || tx0 + lx >= W) continue;
    const int p = static_cast<int>(img0 + static_cast<long long>(ty0 + ly) * W + tx0 + lx);
    const uint8_t cl = s_cls[i];
    ws.cls[p] = cl;
    if (cl) {
      const int r = canny_find(s_lab, i);
      ws.label[p] = static_cast<int>(img0 + static_cast<long long>(ty0 + r / T) * W + tx0 + r % T);
      ws.flag[p] = 0;
    }
  }
}

// One thread per tile-border pixel (top row, left and right columns): joins it with its backward neighbours (left, up-left,
// up, up-right) that lie in another tile.  Every 8-adjacent pair is the backward pair of exactly one of its two pixels.
static __global__ void __launch_bounds__(128) canny_merge_kernel(int H, int W, CannyWs ws) {
  constexpr int T = CANNY_TILE;
  const int t = threadIdx.x;
  int ly, lx;
  if (t < T) { ly = 0; lx = t; }
  else if (t < 2 * T - 1) { ly = t - T + 1; lx = 0; }
  else if (t < 3 * T - 2) { ly = t - 2 * T + 2; lx = T - 1; }
  else return;
  const int gy = blockIdx.y * T + ly, gx = blockIdx.x * T + lx;
  if (gy >= H || gx >= W) return;
  const int p = static_cast<int>((static_cast<long long>(blockIdx.z) * H + gy) * W + gx);
  if (!ws.cls[p]) return;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int oy = k == 0 ? 0 : -1, ox = k == 0 ? -1 : k - 2;
    const int ny = gy + oy, nx = gx + ox;
    if (ny < 0 || nx < 0 || nx >= W) continue;
    if (ny / T == static_cast<int>(blockIdx.y) && nx / T == static_cast<int>(blockIdx.x)) continue;   // joined by the tile
    const int q = p + oy * W + ox;
    if (ws.cls[q]) canny_union(ws.label, p, q);
  }
}

static __global__ void __launch_bounds__(CANNY_THREADS) canny_mark_kernel(int n, CannyWs ws) {
  const int p = blockIdx.x * CANNY_THREADS + threadIdx.x;
  if (p >= n) return;
  const uint8_t cl = ws.cls[p];
  if (!cl) return;
  const int r = canny_find(ws.label, p);
  ws.label[p] = r;            // stays a valid ancestor for concurrent walks
  if (cl == 2) ws.flag[r] = 1;
}

// 16 pixels (48 output bytes) per thread
static __global__ void __launch_bounds__(CANNY_THREADS) canny_out_kernel(int n, CannyWs ws, uint8_t* __restrict__ out) {
  const long long p0 = (static_cast<long long>(blockIdx.x) * CANNY_THREADS + threadIdx.x) * 16;
  if (p0 >= n) return;
  const int cnt = static_cast<int>(min(16ll, n - p0));
  const uint4 c4 = *reinterpret_cast<const uint4*>(ws.cls + p0);   // the class array is padded to 16 bytes
  const uint32_t cw[4] = {c4.x, c4.y, c4.z, c4.w};
  uint32_t v[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const bool cand = k < cnt && ((cw[k / 4] >> (8 * (k % 4))) & 0xffu);
    v[k] = cand && ws.flag[ws.label[p0 + k]] ? 0xffu : 0u;
  }
  uint32_t w[12];
#pragma unroll
  for (int j = 0; j < 12; ++j) {
    uint32_t u = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) u |= v[(4 * j + k) / 3] << (8 * k);
    w[j] = u;
  }
  uint8_t* o = out + p0 * 3;
  if (cnt == 16 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    st16(o, make_uint4(w[0], w[1], w[2], w[3]));
    st16(o + 16, make_uint4(w[4], w[5], w[6], w[7]));
    st16(o + 32, make_uint4(w[8], w[9], w[10], w[11]));
  } else {
#pragma unroll
    for (int j = 0; j < 48; ++j)
      if (j < 3 * cnt) o[j] = static_cast<uint8_t>(v[j / 3]);
  }
}

// Thresholds as cv2.Canny uses them: floored, ordered; magnitudes lie in [0, 2040], so clamping to [-1, 2041] is exact.
inline void canny_thresholds(float low, float high, int* lo, int* hi) {
  double l = std::floor(static_cast<double>(low)), h = std::floor(static_cast<double>(high));
  if (l > h) std::swap(l, h);
  *lo = static_cast<int>(std::min(std::max(l, -1.0), 2041.0));
  *hi = static_cast<int>(std::min(std::max(h, -1.0), 2041.0));
}

// x, out: [B, H, W, 3] uint8 device pointers; ws: canny_workspace_bytes(B*H*W) bytes.  Four launches on `st`.
inline void launch_canny(const uint8_t* x, int B, int H, int W, float low, float high, uint8_t* out, void* ws_base,
                         cudaStream_t st) {
  const long long n = static_cast<long long>(B) * H * W;
  I2IT_CHECK(n < (1ll << 31), "canny: batch*H*W must be below 2^31 (int32 labels)");
  const dim3 tiles((W + CANNY_TILE - 1) / CANNY_TILE, (H + CANNY_TILE - 1) / CANNY_TILE, B);
  I2IT_CHECK(tiles.y <= 65535 && tiles.z <= 65535, "canny: H must be below 2^21 and batch below 65536");
  int lo, hi;
  canny_thresholds(low, high, &lo, &hi);
  const CannyWs ws = canny_ws(ws_base, n);
  const int ni = static_cast<int>(n);
  canny_tile_kernel<<<tiles, CANNY_THREADS, 0, st>>>(x, H, W, lo, hi, ws);
  canny_merge_kernel<<<tiles, 128, 0, st>>>(H, W, ws);
  canny_mark_kernel<<<static_cast<unsigned>((n + CANNY_THREADS - 1) / CANNY_THREADS), CANNY_THREADS, 0, st>>>(ni, ws);
  canny_out_kernel<<<static_cast<unsigned>(((n + 15) / 16 + CANNY_THREADS - 1) / CANNY_THREADS), CANNY_THREADS, 0, st>>>(ni, ws, out);
  I2IT_CUDA(cudaGetLastError());
}

}  // namespace i2it
