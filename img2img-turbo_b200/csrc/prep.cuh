// Load-time weight preparation as a JOB TABLE: every weight / bias of a plan is described by one PrepJob, the table is
// uploaded once and ONE kernel launch folds, re-lays-out and rounds all of them (a second, tiny one runs the
// time-embedding GEMVs).  Round 1 issued ~970 per-tensor launches per engine build; this is 4-5.
//
// Per output element:  v = scale * ( c0*W0[o,i,t] + c1*W1[o,i,t] + sum_a s_a * sum_r B_a[o,r] * A_a[r,i,t] )   in fp32,
// one rounding to the activation dtype.  Replaces peft's runtime LoRA branches (y = Wx + s*B(A(x)), ~1000 extra
// kernels per forward in the reference: /root/reference/src/pix2pix_turbo.py:67-78,137-151,
// /root/reference/src/cyclegan_turbo.py:48-106) and TwinConv (/root/reference/src/pix2pix_turbo.py:16-26).
#pragma once
#include "common.cuh"

namespace i2it {

constexpr int PREP_MAX_ADAPTERS = 4;
constexpr int PREP_ELEMS_PER_BLOCK = 1024;   // 256 threads x 4

enum PrepMode : int {
  PREP_STORE = 0,      // out[tap][row_map(o)][cin_pad]                        (conv / linear weights, GEGLU interleave)
  PREP_SUBPIXEL = 1,   // out[phase*4 + ty*2+tx][o][cin_pad]: pre-summed 2x2 taps of nearest-2x + conv3x3
  PREP_IM2COL3 = 2,    // out[o][32], k = tap*3 + c                             (encoder.conv_in over 3 channels)
  PREP_BIAS = 4,       // outf[row_map(o)] = c0*b[o] + c1*b1[o] + add[o]           (fp32; b1 = w1: TwinConv bias blend)
};

struct PrepJob {
  const float* w0; const float* w1;            // base weight (+ TwinConv partner), PyTorch layout [cout][cin][taps]
  float c0, c1;
  int n_adapters;
  const float* A[PREP_MAX_ADAPTERS];           // [rank][cin*taps]
  const float* B[PREP_MAX_ADAPTERS];           // [cout][rank]
  float s[PREP_MAX_ADAPTERS];
  int rank[PREP_MAX_ADAPTERS];
  void* out;                                   // 16-bit (modes 0-2) or fp32 (mode 4)
  const float* bias; const float* bias_add;    // mode 4
  int mode, cout, cin, taps, cin_pad, rows_total, row_off, interleave_half;
  float scale;
  long long n;                                 // output elements of this job
  long long block0;                            // first block of this job in the launch
};

// folded fp32 value of source element (o, ci, t)
__device__ __forceinline__ float prep_fold(const PrepJob& j, int o, int ci, int t) {
  const long long inner = static_cast<long long>(j.cin) * j.taps;
  const long long src = (static_cast<long long>(o) * j.cin + ci) * j.taps + t;
  float v = j.c0 * j.w0[src];
  if (j.w1) v += j.c1 * j.w1[src];
  const long long jj = static_cast<long long>(ci) * j.taps + t;
  for (int a = 0; a < j.n_adapters; ++a) {
    float d = 0.f;
    const float* Bm = j.B[a] + static_cast<long long>(o) * j.rank[a];
    const float* Am = j.A[a] + jj;
    for (int r = 0; r < j.rank[a]; ++r) d += Bm[r] * Am[r * inner];
    v += j.s[a] * d;
  }
  return v;
}

template <typename T>
__global__ void prep_jobs_kernel(const PrepJob* __restrict__ jobs, int njobs) {
  // locate this block's job (block0 is ascending): binary search, result shared by the block
  __shared__ int s_job;
  if (threadIdx.x == 0) {
    int lo = 0, hi = njobs - 1;
    const long long b = blockIdx.x;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (jobs[mid].block0 <= b) lo = mid; else hi = mid - 1;
    }
    s_job = lo;
  }
  __syncthreads();
  const PrepJob& j = jobs[s_job];
  const long long base = (static_cast<long long>(blockIdx.x) - j.block0) * PREP_ELEMS_PER_BLOCK;
#pragma unroll 1
  for (int e = 0; e < PREP_ELEMS_PER_BLOCK / 256; ++e) {
    const long long i = base + e * 256 + threadIdx.x;
    if (i >= j.n) return;
    if (j.mode == PREP_STORE) {
      const int ci = static_cast<int>(i % j.cin_pad);
      long long r = i / j.cin_pad;
      const int o = static_cast<int>(r % j.cout);
      const int t = static_cast<int>(r / j.cout);
      int orow = o;
      if (j.interleave_half > 0) orow = (o < j.interleave_half) ? 2 * o : 2 * (o - j.interleave_half) + 1;
      orow += j.row_off;
      const float v = (ci < j.cin) ? prep_fold(j, o, ci, t) * j.scale : 0.f;
      reinterpret_cast<T*>(j.out)[(static_cast<long long>(t) * j.rows_total + orow) * j.cin_pad + ci] = Elem<T>::from_f(v);
    } else if (j.mode == PREP_SUBPIXEL) {
      // rows R(0,0)={0} R(0,1)={1,2} R(1,0)={0,1} R(1,1)={2} (same for columns); summed in fp32, rounded once
      const int ci = static_cast<int>(i % j.cin_pad);
      long long r = i / j.cin_pad;
      const int o = static_cast<int>(r % j.cout);
      const int t16 = static_cast<int>(r / j.cout);
      const int phase = t16 >> 2, ty = (t16 >> 1) & 1, tx = t16 & 1, py = phase >> 1, px = phase & 1;
      float v = 0.f;
      if (ci < j.cin) {
        const int ky0 = (py == 0) ? (ty == 0 ? 0 : 1) : (ty == 0 ? 0 : 2), ky1 = (py == 0) ? (ty == 0 ? 0 : 2) : (ty == 0 ? 1 : 2);
        const int kx0 = (px == 0) ? (tx == 0 ? 0 : 1) : (tx == 0 ? 0 : 2), kx1 = (px == 0) ? (tx == 0 ? 0 : 2) : (tx == 0 ? 1 : 2);
        for (int ky = ky0; ky <= ky1; ++ky)
          for (int kx = kx0; kx <= kx1; ++kx) v += prep_fold(j, o, ci, ky * 3 + kx);
      }
      reinterpret_cast<T*>(j.out)[i] = Elem<T>::from_f(v * j.scale);
    } else if (j.mode == PREP_IM2COL3) {
      const int o = static_cast<int>(i / 32), k = static_cast<int>(i % 32);
      float v = 0.f;
      if (k < 27) v = prep_fold(j, o, k % 3, k / 3);
      reinterpret_cast<T*>(j.out)[i] = Elem<T>::from_f(v * j.scale);
    } else {   // PREP_BIAS
      const int o = static_cast<int>(i);
      int orow = o;
      if (j.interleave_half > 0) orow = (o < j.interleave_half) ? 2 * o : 2 * (o - j.interleave_half) + 1;
      reinterpret_cast<float*>(j.out)[orow + j.row_off] =
          (j.bias ? j.c0 * j.bias[o] : 0.f) + (j.w1 ? j.c1 * j.w1[o] : 0.f) + (j.bias_add ? j.bias_add[o] : 0.f);
    }
  }
}

// y = act(W' x + b) with W' folded on the fly (fp32), one warp per output row; several independent GEMVs per launch
// (the time-embedding MLP at t == 999 and every resnet's time_emb_proj: computed once per finalize).
struct GemvJob {
  const float* w; const float* b; const float* x; float* y;
  int n_adapters;
  const float* A[PREP_MAX_ADAPTERS]; const float* B[PREP_MAX_ADAPTERS];
  float s[PREP_MAX_ADAPTERS]; int rank[PREP_MAX_ADAPTERS];
  int out, in, silu_out;
  int warp0;                                   // first warp of this job in the launch
};

static __global__ void gemv_jobs_kernel(const GemvJob* __restrict__ jobs, int njobs) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  int lo = 0, hi = njobs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].warp0 <= gw) lo = mid; else hi = mid - 1;
  }
  const GemvJob& j = jobs[lo];
  const int o = gw - j.warp0;
  if (o >= j.out) return;
  float a = 0.f;
  for (int i = lane; i < j.in; i += 32) {
    float w = j.w[static_cast<long long>(o) * j.in + i];
    for (int ad = 0; ad < j.n_adapters; ++ad) {
      float d = 0.f;
      for (int r = 0; r < j.rank[ad]; ++r) d += j.B[ad][o * j.rank[ad] + r] * j.A[ad][static_cast<long long>(r) * j.in + i];
      w += j.s[ad] * d;
    }
    a += w * j.x[i];
  }
  a = warp_sum(a);
  if (lane == 0) {
    a += j.b ? j.b[o] : 0.f;
    j.y[o] = j.silu_out ? a / (1.f + expf(-a)) : a;   // exact SiLU: load-time only
  }
}

}  // namespace i2it
