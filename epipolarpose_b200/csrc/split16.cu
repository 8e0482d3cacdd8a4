// Element-wise producers / consumers of split-fp16 tensors (include/epb.h, "f16x3" family):
//   x * s = hi + lo,  hi = fp16(x*s), lo = fp16(x*s - hi), two planes [2][rows][C].
// Reference call sites: the BatchNorm2d / ReLU / residual add / MaxPool2d / AvgPool2d of
// lib/models/pose3d_resnet.py:24,31-47,56-88,101-103,125,134,179,187-189,208 and their
// autograd.  Every kernel is one HBM pass: fp32 rows in, two fp16 planes out (the same
// 4 bytes per element as an fp32 store), so that the tensor-core kernels (conv16.cu,
// wgrad16.cu) can take their operands by TMA with no transformation.
// `planes` (1 or 2) is the plane count of the split tensors a kernel writes or reads: with 1
// (the single-pass "f16" mode) only the hi plane exists, [1][rows][C], and nothing is written
// where the lo plane would lie; the hi plane is the same either way.
#include <cuda_fp16.h>
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr float kHalfMax = 65504.f;

// (a, b) * s -> packed fp16 pairs hi, lo
__device__ __forceinline__ void split2(float a, float b, float s, uint32_t& hi, uint32_t& lo) {
  a = fminf(fmaxf(a * s, -kHalfMax), kHalfMax);
  b = fminf(fmaxf(b * s, -kHalfMax), kHalfMax);
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void split8(const float (&v)[8], float s, uint4& hi, uint4& lo) {
  split2(v[0], v[1], s, hi.x, lo.x);
  split2(v[2], v[3], s, hi.y, lo.y);
  split2(v[4], v[5], s, hi.z, lo.z);
  split2(v[6], v[7], s, hi.w, lo.w);
}
__device__ __forceinline__ float2 h2f(uint32_t u) {
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
// 8 values (hi + lo) * inv
__device__ __forceinline__ void join8(uint4 hi, uint4 lo, float inv, float (&v)[8]) {
  const uint32_t* H = &hi.x;
  const uint32_t* L = &lo.x;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 a = h2f(H[k]), b = h2f(L[k]);
    v[2 * k] = (a.x + b.x) * inv;
    v[2 * k + 1] = (a.y + b.y) * inv;
  }
}
__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
  const float4 a = ldg_stream(reinterpret_cast<const float4*>(p));
  const float4 b = ldg_stream(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ld8c(const float* p, float (&v)[8]) {   // cached (per-channel vectors)
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

inline int ew_blocks(int64_t items) {
  int64_t b = (items + kThreads - 1) / kThreads;
  const int64_t cap = (int64_t)kNumSMs * 16;
  return (int)(b < cap ? (b > 0 ? b : 1) : cap);
}

// ------------------------------------------------------------------ forward
__global__ void __launch_bounds__(kThreads)
bn_act_split_kernel(const float* __restrict__ x, const float* __restrict__ scale,
                    const float* __restrict__ shift, const float* __restrict__ r,
                    const float* __restrict__ rscale, const float* __restrict__ rshift,
                    const uint4* __restrict__ rs, const float* __restrict__ rs_sc, int relu,
                    int64_t total8, int C8, uint4* __restrict__ y, const float* __restrict__ y_sc,
                    uint8_t* __restrict__ mask_bits, int planes) {
  const float s = y_sc[0];
  const float rinv = rs ? rs_sc[1] : 0.f;
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < total8;
       i += (int64_t)gridDim.x * kThreads) {
    const int c = (int)(i % C8) * 8;
    float v[8];
    ld8(x + i * 8, v);
    if (scale) {
      float sc[8], sh[8];
      ld8c(scale + c, sc);
      ld8c(shift + c, sh);
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = fmaf(v[k], sc[k], sh[k]);
    }
    if (r) {
      float q[8];
      ld8(r + i * 8, q);
      if (rscale) {
        float sc[8], sh[8];
        ld8c(rscale + c, sc);
        ld8c(rshift + c, sh);
#pragma unroll
        for (int k = 0; k < 8; ++k) q[k] = fmaf(q[k], sc[k], sh[k]);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] += q[k];
    } else if (rs) {
      float q[8];
      join8(rs[i], planes == 2 ? rs[total8 + i] : make_uint4(0u, 0u, 0u, 0u), rinv, q);
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] += q[k];
    }
    if (mask_bits) {                          // bit k of byte i: element 8*i + k passes the ReLU
      unsigned bits = 0;
#pragma unroll
      for (int k = 0; k < 8; ++k) bits |= (v[k] > 0.f ? 1u : 0u) << k;
      mask_bits[i] = (uint8_t)bits;
    }
    if (relu) {
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = fmaxf(v[k], 0.f);
    }
    uint4 hi, lo;
    split8(v, s, hi, lo);
    y[i] = hi;
    if (planes == 2) y[total8 + i] = lo;
  }
}

__global__ void __launch_bounds__(kThreads)
bn_relu_maxpool_split_kernel(const float* __restrict__ x, const float* __restrict__ scale,
                             const float* __restrict__ shift, uint4* __restrict__ y,
                             const float* __restrict__ y_sc, uint2* __restrict__ argidx, int N, int H,
                             int W, int C8, int planes) {
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  const int64_t total = (int64_t)N * Ho * Wo * C8;
  const float s = y_sc[0];
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * kThreads) {
    const int c8 = (int)(i % C8);
    int64_t p = i / C8;
    const int ow = (int)(p % Wo); p /= Wo;
    const int oh = (int)(p % Ho);
    const int n = (int)(p / Ho);
    float sc[8], sh[8], best[8];
    unsigned char bi[8];
    ld8c(scale + c8 * 8, sc);
    ld8c(shift + c8 * 8, sh);
#pragma unroll
    for (int k = 0; k < 8; ++k) { best[k] = -INFINITY; bi[k] = 0; }
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int ih = oh * 2 - 1 + kh;
      if (ih < 0 || ih >= H) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int iw = ow * 2 - 1 + kw;
        if (iw < 0 || iw >= W) continue;
        float v[8];
        ld8c(x + (((int64_t)(n * H + ih) * W + iw) * C8 + c8) * 8, v);
        const unsigned char me = (unsigned char)(kh * 3 + kw);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float a = fmaxf(fmaf(v[k], sc[k], sh[k]), 0.f);
          if (a > best[k]) { best[k] = a; bi[k] = me; }
        }
      }
    }
    uint4 hi, lo;
    split8(best, s, hi, lo);
    y[i] = hi;
    if (planes == 2) y[total + i] = lo;
    if (argidx) {
      uint2 a;
      a.x = bi[0] | (bi[1] << 8) | (bi[2] << 16) | ((unsigned)bi[3] << 24);
      a.y = bi[4] | (bi[5] << 8) | (bi[6] << 16) | ((unsigned)bi[7] << 24);
      argidx[i] = a;
    }
  }
}

// one thread = 8 consecutive k of one patch row; the (channel, tap) decomposition of k is a
// per-CTA lookup table (no integer divisions per element)
__global__ void __launch_bounds__(kThreads)
im2col_split_kernel(const float* __restrict__ img, uint4* __restrict__ col,
                    const float* __restrict__ col_sc, int N, int C, int Hi, int Wi, int kh, int kw,
                    int stride, int pad, int Ho, int Wo, int Kpad, int planes) {
  extern __shared__ int lut[];                 // [Kpad]: (c*Hi + r)*Wi + s | r << 24 ... packed below
  int* off = lut;                              // element offset of (c, r, s) relative to (ih0, iw0)
  int* rs = lut + Kpad;                        // r << 16 | s ; -1 for padding columns
  const int K = kh * kw * C;
  for (int kk = threadIdx.x; kk < Kpad; kk += kThreads) {
    if (kk < K) {
      const int t = kk / C, c = kk - t * C;
      const int r = t / kw, sx = t - r * kw;
      off[kk] = (c * Hi + r) * Wi + sx;
      rs[kk] = (r << 16) | sx;
    } else {
      off[kk] = 0;
      rs[kk] = -1;
    }
  }
  __syncthreads();
  const int K8 = Kpad >> 3;
  const int64_t total = (int64_t)N * Ho * Wo * K8;
  const float s = col_sc[0];
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * kThreads) {
    const int k8 = (int)(i % K8);
    int64_t m = i / K8;
    const int ow = (int)(m % Wo); m /= Wo;
    const int oh = (int)(m % Ho);
    const int n = (int)(m / Ho);
    const int ih0 = oh * stride - pad, iw0 = ow * stride - pad;
    const float* base = img + (int64_t)n * C * Hi * Wi + (int64_t)ih0 * Wi + iw0;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int kk = k8 * 8 + e;
      const int q = rs[kk];
      const int ih = ih0 + (q >> 16), iw = iw0 + (q & 0xffff);
      v[e] = (q >= 0 && ih >= 0 && ih < Hi && iw >= 0 && iw < Wi) ? __ldg(base + off[kk]) : 0.f;
    }
    uint4 hi, lo;
    split8(v, s, hi, lo);
    col[i] = hi;
    if (planes == 2) col[total + i] = lo;
  }
}

// Same matrix, staged: a CTA takes kSeg consecutive output pixels of one output row, loads the
// C x kh x (stride*(kSeg-1)+kw) input window once (coalesced rows, zero outside the image) and builds
// its kSeg patch rows from shared memory -- every input pixel is read from HBM/L2 once per CTA instead
// of once per tap that touches it.
constexpr int kSeg = 64;
__global__ void __launch_bounds__(kThreads)
im2col_split_tiled_kernel(const float* __restrict__ img, uint4* __restrict__ col,
                          const float* __restrict__ col_sc, int N, int C, int Hi, int Wi, int kh, int kw,
                          int stride, int pad, int Ho, int Wo, int Kpad, int segs, int tw, int planes) {
  extern __shared__ int smi[];
  int* lut = smi;                               // [8][Kpad/8]: window offset of (c, r, s), -1 for padding columns
  float* win = reinterpret_cast<float*>(smi + Kpad);        // [C][kh][tw]
  const int K = kh * kw * C;
  int b = blockIdx.x;
  const int seg = b % segs; b /= segs;
  const int oh = b % Ho;
  const int n = b / Ho;
  const int ow0 = seg * kSeg;
  const int ih0 = oh * stride - pad, iw0 = ow0 * stride - pad;
  for (int kk = threadIdx.x; kk < Kpad; kk += kThreads) {
    int o = -1;
    if (kk < K) {
      const int t = kk / C, c = kk - t * C;
      const int r = t / kw, sx = t - r * kw;
      o = (c * kh + r) * tw + sx;
    }
    lut[(kk & 7) * (Kpad >> 3) + (kk >> 3)] = o;       // [e][k8]: a warp's lanes (consecutive k8) hit distinct banks
  }
  const int wsize = C * kh * tw;
  for (int i = threadIdx.x; i < wsize; i += kThreads) {
    const int x = i % tw;
    const int cr = i / tw;
    const int r = cr % kh, c = cr / kh;
    const int ih = ih0 + r, iw = iw0 + x;
    float v = 0.f;
    if (ih >= 0 && ih < Hi && iw >= 0 && iw < Wi) v = __ldg(img + (((int64_t)n * C + c) * Hi + ih) * Wi + iw);
    win[i] = v;
  }
  __syncthreads();
  const int K8 = Kpad >> 3;
  const int npx = min(kSeg, Wo - ow0);
  const int64_t total = (int64_t)N * Ho * Wo * K8;
  const int64_t row0 = (((int64_t)n * Ho + oh) * Wo + ow0) * K8;
  const float s = col_sc[0];
  for (int it = threadIdx.x; it < npx * K8; it += kThreads) {
    const int p = it / K8, k8 = it - p * K8;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int o = lut[e * K8 + k8];
      v[e] = o >= 0 ? win[o + p * stride] : 0.f;
    }
    uint4 hi, lo;
    split8(v, s, hi, lo);
    col[row0 + it] = hi;
    if (planes == 2) col[total + row0 + it] = lo;
  }
}

// ------------------------------------------------------------------ batched fp32 -> split
__device__ __forceinline__ const epb_split_job& find_job(const epb_split_job* jobs, int njobs,
                                                         int& idx) {
  int lo = 0, hi = njobs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].first_block <= (long long)blockIdx.x) lo = mid;
    else hi = mid - 1;
  }
  idx = lo;
  return jobs[lo];
}

__global__ void __launch_bounds__(kThreads)
split_amax_kernel(const epb_split_job* __restrict__ jobs, int njobs, uint32_t* __restrict__ amax) {
  int ji;
  const epb_split_job j = find_job(jobs, njobs, ji);
  const int64_t i0 = ((int64_t)blockIdx.x - j.first_block) * 2048;
  const int64_t i1 = i0 + 2048 < j.n ? i0 + 2048 : j.n;
  float m = 0.f;
  for (int64_t i = i0 + threadIdx.x; i < i1; i += kThreads) m = fmaxf(m, fabsf(j.src[i]));
  m = warp_max(m);
  __shared__ float sm[kThreads / 32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kThreads / 32; ++w) m = fmaxf(m, sm[w]);
    if (m > 0.f) atomicMax(amax + ji, __float_as_uint(m));   // non-negative floats order as uints
  }
}

// scale 2^(13 - floor(log2(amax))): the largest scaled magnitude lies in [2^13, 2^14)
__device__ __forceinline__ float pow2_scale(float amax) {
  if (!(amax > 0.f) || !isfinite(amax)) return 1.f;
  int e;
  frexpf(amax, &e);                 // amax = f * 2^e, f in [0.5, 1)  ->  floor(log2) = e - 1
  int k = 13 - (e - 1);
  k = k < -100 ? -100 : (k > 100 ? 100 : k);
  return ldexpf(1.f, k);
}

__global__ void __launch_bounds__(kThreads)
split_apply_kernel(const epb_split_job* __restrict__ jobs, int njobs,
                   const uint32_t* __restrict__ amax, int planes) {
  int ji;
  const epb_split_job j = find_job(jobs, njobs, ji);
  const float s = pow2_scale(__uint_as_float(amax[ji]));
  const int64_t i0 = ((int64_t)blockIdx.x - j.first_block) * 2048;
  if (i0 == 0 && threadIdx.x == 0) {
    j.sc[0] = s;
    j.sc[1] = 1.f / s;
  }
  const int64_t i1 = i0 + 2048 < j.n ? i0 + 2048 : j.n;
  __half* hi = reinterpret_cast<__half*>(j.dst);
  __half* lo = hi + j.n;
  for (int64_t i = i0 + threadIdx.x; i < i1; i += kThreads) {
    const float v = j.src[i] * s;
    const __half h = __float2half_rn(v);
    hi[i] = h;
    if (planes == 2) lo[i] = __float2half_rn(v - __half2float(h));
  }
}

// single tensor, pointers as kernel arguments (no device job table: usable on tensors whose
// address is only known at call time, e.g. the logit gradient handed over by autograd)
__global__ void __launch_bounds__(kThreads)
split_amax_one_kernel(const float4* __restrict__ src, int64_t n4, uint32_t* __restrict__ amax) {
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n4; i += (int64_t)gridDim.x * kThreads) {
    const float4 v = ldg_stream(src + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  m = warp_max(m);
  __shared__ float sm[kThreads / 32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kThreads / 32; ++w) m = fmaxf(m, sm[w]);
    if (m > 0.f) atomicMax(amax, __float_as_uint(m));
  }
}

__global__ void __launch_bounds__(kThreads)
split_apply_one_kernel(const float4* __restrict__ src, int64_t n4, const uint32_t* __restrict__ amax,
                       uint2* __restrict__ dst, float* __restrict__ sc, int planes) {
  const float s = pow2_scale(__uint_as_float(*amax));
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    sc[0] = s;
    sc[1] = 1.f / s;
  }
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n4; i += (int64_t)gridDim.x * kThreads) {
    const float4 v = ldg_stream(src + i);
    uint2 hi, lo;
    split2(v.x, v.y, s, hi.x, lo.x);
    split2(v.z, v.w, s, hi.y, lo.y);
    dst[i] = hi;
    if (planes == 2) dst[n4 + i] = lo;
  }
}

// ------------------------------------------------------------------ BatchNorm backward

struct RowMap {
  int C4, tpr, rpi, chunks;
};
inline RowMap make_rowmap(int C) {
  RowMap r;
  r.C4 = C / 4;
  r.tpr = r.C4 < kThreads ? r.C4 : kThreads;
  r.rpi = kThreads / r.tpr;
  if (r.rpi < 1) r.rpi = 1;
  r.chunks = (r.C4 + r.tpr - 1) / r.tpr;
  return r;
}

__device__ __forceinline__ float4 mask4(float4 dy, float4 xv, const uint2* mask_hi, int64_t i,
                                        float4 s, float4 b, int relu) {
  if (mask_hi) {
    const uint2 m = mask_hi[i];            // 4 fp16 values of the (non-negative) block output
    return make_float4((m.x & 0x7fffu) ? dy.x : 0.f, (m.x & 0x7fff0000u) ? dy.y : 0.f,
                       (m.y & 0x7fffu) ? dy.z : 0.f, (m.y & 0x7fff0000u) ? dy.w : 0.f);
  }
  if (relu) {
    return make_float4(fmaf(xv.x, s.x, b.x) > 0.f ? dy.x : 0.f, fmaf(xv.y, s.y, b.y) > 0.f ? dy.y : 0.f,
                       fmaf(xv.z, s.z, b.z) > 0.f ? dy.z : 0.f, fmaf(xv.w, s.w, b.w) > 0.f ? dy.w : 0.f);
  }
  return dy;
}

// Pass 1: per-CTA partial reductions.  CTA (w, chunk) folds rows (w + k*gridDim.x)*rpi + slot
// into registers and stores FOUR per-channel partials (sum g, sum g*xhat, max|g|, max|xhat|)
// to parts[(v*W + w)*C + c] -- no atomics: the second pass adds them in a fixed order, so the
// parameter gradients and the scale of dz are run-to-run identical.
// mask of element quad i: MASK 1 = four fp16 values of the block output's hi plane, MASK 2 = four bits
// (low / high nibble of byte i/2 of the bit mask bn_act_split wrote)
template <int MASK>
__device__ __forceinline__ uint2 load_mask(const uint2* mask, int64_t i) {
  if (MASK == 1) return __ldg(mask + i);
  const unsigned byte = __ldg(reinterpret_cast<const uint8_t*>(mask) + (i >> 1));
  return make_uint2((i & 1) ? (byte >> 4) : (byte & 15u), 0u);
}

template <int MASK>
__global__ void __launch_bounds__(kThreads, 3)
bn_bwd_partial_kernel(const float4* __restrict__ dy, const float4* __restrict__ x,
                      const uint2* __restrict__ mask_hi, const float4* __restrict__ scale,
                      const float4* __restrict__ shift, const float4* __restrict__ mean,
                      const float4* __restrict__ invstd, int relu, int64_t M, int C, RowMap rm,
                      float* __restrict__ parts, uint32_t* __restrict__ bound_bits) {
  if (bound_bits && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *bound_bits = 0u;
  const int slot = threadIdx.x / rm.tpr, tin = threadIdx.x % rm.tpr;
  const int c4 = blockIdx.y * rm.tpr + tin;
  const bool active = (c4 < rm.C4) && (slot < rm.rpi);
  const int64_t nblk = (M + rm.rpi - 1) / rm.rpi;
  float4 acc[4] = {{0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}, {0, 0, 0, 0}};
  if (active) {
    const float4 mu = mean[c4], is = invstd[c4];
    float4 s = make_float4(0, 0, 0, 0), b = s;
    if (!MASK) { s = scale[c4]; b = shift[c4]; }
    auto fold = [&](float4 dv, float4 xv, uint2 mk) {
      float4 g;
      if (MASK == 1) {
        g = make_float4((mk.x & 0x7fffu) ? dv.x : 0.f, (mk.x & 0x7fff0000u) ? dv.y : 0.f,
                        (mk.y & 0x7fffu) ? dv.z : 0.f, (mk.y & 0x7fff0000u) ? dv.w : 0.f);
      } else if (MASK == 2) {                 // mk.x = this quad's four bits
        g = make_float4((mk.x & 1u) ? dv.x : 0.f, (mk.x & 2u) ? dv.y : 0.f,
                        (mk.x & 4u) ? dv.z : 0.f, (mk.x & 8u) ? dv.w : 0.f);
      } else {
        g = mask4(dv, xv, nullptr, 0, s, b, relu);
      }
      const float4 xh = make_float4((xv.x - mu.x) * is.x, (xv.y - mu.y) * is.y,
                                    (xv.z - mu.z) * is.z, (xv.w - mu.w) * is.w);
      acc[0].x += g.x; acc[0].y += g.y; acc[0].z += g.z; acc[0].w += g.w;
      acc[1].x += g.x * xh.x; acc[1].y += g.y * xh.y; acc[1].z += g.z * xh.z; acc[1].w += g.w * xh.w;
      acc[2].x = fmaxf(acc[2].x, fabsf(g.x)); acc[2].y = fmaxf(acc[2].y, fabsf(g.y));
      acc[2].z = fmaxf(acc[2].z, fabsf(g.z)); acc[2].w = fmaxf(acc[2].w, fabsf(g.w));
      acc[3].x = fmaxf(acc[3].x, fabsf(xh.x)); acc[3].y = fmaxf(acc[3].y, fabsf(xh.y));
      acc[3].z = fmaxf(acc[3].z, fabsf(xh.z)); acc[3].w = fmaxf(acc[3].w, fabsf(xh.w));
    };
    int64_t blk = blockIdx.x;
    const int64_t step = gridDim.x;
    for (; blk + 3 * step < nblk; blk += 4 * step) {       // four rows per trip: 8-12 loads in flight
      float4 xv[4], dv[4];
      uint2 mk[4];
      bool ok[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t r = (blk + u * step) * rm.rpi + slot;
        ok[u] = r < M;
        mk[u] = make_uint2(0u, 0u);
        if (ok[u]) {
          const int64_t i = r * rm.C4 + c4;
          xv[u] = ldg_stream(x + i);
          dv[u] = ldg_stream(dy + i);
          if (MASK) mk[u] = load_mask<MASK>(mask_hi, i);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (ok[u]) fold(dv[u], xv[u], mk[u]);
    }
    for (; blk < nblk; blk += step) {
      const int64_t r = blk * rm.rpi + slot;
      if (r >= M) break;
      const int64_t i = r * rm.C4 + c4;
      const float4 xv = ldg_stream(x + i);
      const float4 dv = ldg_stream(dy + i);
      fold(dv, xv, MASK ? load_mask<MASK>(mask_hi, i) : make_uint2(0u, 0u));
    }
  }
  __shared__ float4 sh[4][kThreads];
#pragma unroll
  for (int v = 0; v < 4; ++v) sh[v][threadIdx.x] = acc[v];
  __syncthreads();
  if (slot == 0 && active) {
    const int64_t W = gridDim.x;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      float4 t = sh[v][tin];
      for (int q = 1; q < rm.rpi; ++q) {
        const float4 u = sh[v][q * rm.tpr + tin];
        if (v < 2) { t.x += u.x; t.y += u.y; t.z += u.z; t.w += u.w; }
        else { t.x = fmaxf(t.x, u.x); t.y = fmaxf(t.y, u.y); t.z = fmaxf(t.z, u.z); t.w = fmaxf(t.w, u.w); }
      }
      *reinterpret_cast<float4*>(parts + ((int64_t)v * W + blockIdx.x) * C + c4 * 4) = t;
    }
  }
}

// Pass 2: 8 channels per CTA (one 32-byte sector per row), 32 groups of partials per channel, every
// group and then the groups added in a fixed order.
//   coef == NULL : sums[0..2C) += (sum g, sum g*xhat), maxes = max(maxes, ...)   (epb_bn_bwd_reduce_mx)
//   coef != NULL : coef[0..2C) = (k1 = sum_g/M, k2 = sum_gx/M), parameter gradients, and the bound
//     |dz_c| <= |gamma_c*invstd_c| * (max|g|_c + |k1_c| + max|xhat|_c * |k2_c|)  max-ed into *bound_bits
__global__ void __launch_bounds__(256)
bn_bwd_combine_kernel(const float* __restrict__ parts, int W, double M, int C,
                      double* __restrict__ sums, float* __restrict__ maxes, float* __restrict__ coef,
                      const float* __restrict__ gamma, const float* __restrict__ invstd,
                      float* __restrict__ dgamma, float* __restrict__ dbeta,
                      uint32_t* __restrict__ bound_bits) {
  const int ch = threadIdx.x & 7, g = threadIdx.x >> 3;        // 32 groups
  const int c = blockIdx.x * 8 + ch;
  double a0 = 0, a1 = 0;
  float m0 = 0.f, m1 = 0.f;
  if (c < C) {
    const float* p0 = parts + c;
    const int64_t plane = (int64_t)W * C;
    for (int w0 = g; w0 < W; w0 += 32 * 8) {       // batches of 8 rows: 32 independent loads in flight
      float v[4][8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int w = w0 + 32 * u;
        const int64_t o = (int64_t)(w < W ? w : 0) * C;
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k][u] = (w < W) ? __ldg(p0 + k * plane + o) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        a0 += (double)v[0][u];
        a1 += (double)v[1][u];
        m0 = fmaxf(m0, v[2][u]);
        m1 = fmaxf(m1, v[3][u]);
      }
    }
  }
  __shared__ double sa[2][32][8];
  __shared__ float sm[2][32][8];
  sa[0][g][ch] = a0; sa[1][g][ch] = a1;
  sm[0][g][ch] = m0; sm[1][g][ch] = m1;
  __syncthreads();
#pragma unroll
  for (int half = 16; half > 0; half >>= 1) {      // fixed pairing: run-to-run identical
    if (g < half) {
      sa[0][g][ch] += sa[0][g + half][ch];
      sa[1][g][ch] += sa[1][g + half][ch];
      sm[0][g][ch] = fmaxf(sm[0][g][ch], sm[0][g + half][ch]);
      sm[1][g][ch] = fmaxf(sm[1][g][ch], sm[1][g + half][ch]);
    }
    __syncthreads();
  }
  if (g != 0) return;
  a0 = sa[0][0][ch]; a1 = sa[1][0][ch];
  m0 = sm[0][0][ch]; m1 = sm[1][0][ch];
  float bound = 0.f;
  if (c < C) {
    if (!coef) {
      sums[c] += a0;
      sums[C + c] += a1;
      maxes[c] = fmaxf(maxes[c], m0);
      maxes[C + c] = fmaxf(maxes[C + c], m1);
    } else {
      const float k0 = (gamma ? gamma[c] : 1.f) * invstd[c];
      const float k1 = (float)(a0 / M), k2 = (float)(a1 / M);
      coef[c] = k1;
      coef[C + c] = k2;
      if (dgamma) dgamma[c] = (float)a1;
      if (dbeta) dbeta[c] = (float)a0;
      bound = fabsf(k0) * (m0 + fabsf(k1) + m1 * fabsf(k2));
    }
  }
  if (coef) {                                  // threads 0..7 of warp 0
    for (int o = 4; o > 0; o >>= 1) bound = fmaxf(bound, __shfl_xor_sync(0xffu, bound, o));
    if (ch == 0) atomicMax(bound_bits, __float_as_uint(bound));   // order-independent
  }
}

// one CTA: per-channel coefficients (k1 = sum_g/M, k2 = sum_gx/M overwrite maxes[0..2C)),
// parameter gradients, and the power-of-two scale of dz from the bound
//   |dz_c| <= |gamma_c*invstd_c| * (max|g|_c + |k1_c| + max|xhat|_c * |k2_c|)
__global__ void __launch_bounds__(1024)
bn_bwd_coef_split_kernel(const double* __restrict__ sums, float* __restrict__ maxes, double M, int C,
                         const float* __restrict__ gamma, const float* __restrict__ invstd,
                         float* __restrict__ dz_sc, float* __restrict__ dgamma,
                         float* __restrict__ dbeta) {
  float bound = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double sg = sums[c], sgx = sums[C + c];
    const float k0 = (gamma ? gamma[c] : 1.f) * invstd[c];
    const float k1 = (float)(sg / M), k2 = (float)(sgx / M);
    const float mg = maxes[c], mx = maxes[C + c];
    bound = fmaxf(bound, fabsf(k0) * (mg + fabsf(k1) + mx * fabsf(k2)));
    maxes[c] = k1;
    maxes[C + c] = k2;
    if (dgamma) dgamma[c] = (float)sgx;
    if (dbeta) dbeta[c] = (float)sg;
  }
  bound = warp_max(bound);
  __shared__ float sm[32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = bound;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) bound = fmaxf(bound, sm[w]);
    const float s = pow2_scale(bound);
    dz_sc[0] = s;
    dz_sc[1] = 1.f / s;
  }
}

__global__ void __launch_bounds__(kThreads)
bn_bwd_apply_split_kernel(const float4* dy /* may alias dy_masked */, const float4* __restrict__ x,
                          const uint2* __restrict__ mask_hi, const float4* __restrict__ scale,
                          const float4* __restrict__ shift, const float4* __restrict__ mean,
                          const float4* __restrict__ invstd, const float4* __restrict__ gamma,
                          int relu, const float4* __restrict__ k1v, const float4* __restrict__ k2v,
                          uint2* __restrict__ dz, float* __restrict__ dz_sc,
                          const float* __restrict__ bound, float4* dy_masked, int64_t total4, int C4,
                          int mask_bits, int planes) {
  // scale of dz: from the bound the combine pass left (fused entry point), else as published in dz_sc
  const float s = bound ? pow2_scale(*bound) : dz_sc[0];
  if (bound && blockIdx.x == 0 && threadIdx.x == 0) {
    dz_sc[0] = s;
    dz_sc[1] = 1.f / s;
  }
  // two independent elements per trip: six streaming loads in flight per thread
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t i0 = (int64_t)blockIdx.x * kThreads + threadIdx.x; i0 < total4; i0 += 2 * stride) {
    const int64_t idx[2] = {i0, i0 + stride};
    float4 xv[2], dv[2];
    uint2 mk[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (idx[u] < total4) {
        xv[u] = ldg_stream(x + idx[u]);
        dv[u] = __ldcs(dy + idx[u]);
        if (mask_hi) mk[u] = mask_bits ? load_mask<2>(mask_hi, idx[u]) : mask_hi[idx[u]];
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int64_t i = idx[u];
      if (i >= total4) break;
      const int c4 = (int)(i % C4);
      float4 g = dv[u];
      if (mask_hi && mask_bits) {
        g = make_float4((mk[u].x & 1u) ? g.x : 0.f, (mk[u].x & 2u) ? g.y : 0.f,
                        (mk[u].x & 4u) ? g.z : 0.f, (mk[u].x & 8u) ? g.w : 0.f);
      } else if (mask_hi) {
        g = make_float4((mk[u].x & 0x7fffu) ? g.x : 0.f, (mk[u].x & 0x7fff0000u) ? g.y : 0.f,
                        (mk[u].y & 0x7fffu) ? g.z : 0.f, (mk[u].y & 0x7fff0000u) ? g.w : 0.f);
      } else {
        g = mask4(g, xv[u], nullptr, i, scale[c4], shift[c4], relu);
      }
      const float4 mu = mean[c4], is = invstd[c4], b = k1v[c4], c = k2v[c4];
      float4 a = is;
      if (gamma) {
        const float4 ga = gamma[c4];
        a.x *= ga.x; a.y *= ga.y; a.z *= ga.z; a.w *= ga.w;
      }
      float4 o;
      o.x = a.x * (g.x - b.x - (xv[u].x - mu.x) * is.x * c.x);
      o.y = a.y * (g.y - b.y - (xv[u].y - mu.y) * is.y * c.y);
      o.z = a.z * (g.z - b.z - (xv[u].z - mu.z) * is.z * c.z);
      o.w = a.w * (g.w - b.w - (xv[u].w - mu.w) * is.w * c.w);
      uint2 hi, lo;
      split2(o.x, o.y, s, hi.x, lo.x);
      split2(o.z, o.w, s, hi.y, lo.y);
      dz[i] = hi;
      if (planes == 2) dz[total4 + i] = lo;
      if (dy_masked) dy_masked[i] = g;
    }
  }
}

// one CTA: hard bound of a post-activation tensor from the statistics of its conv output(s)
__device__ __forceinline__ float group_bound(const double* stats, const float* scale,
                                             const float* shift, double M, int C) {
  float b = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double mean = stats[c] / M;
    double var = stats[C + c] / M - mean * mean;
    if (var < 0) var = 0;
    const double sc = scale[c], sh = shift[c];
    // no element of a sample lies further than sqrt(M - 1) standard deviations from its mean
    b = fmaxf(b, (float)(fabs(sc * mean + sh) + fabs(sc) * sqrt(M * var)));
  }
  return b;
}

// sc = {s, 1/s, bound, 0}: s the largest power of two with s * bound <= 2^15 (fp16 max is 65504)
__device__ __forceinline__ void publish_act_scale(float b1, float b2, const float* res_sc, float* sc) {
  float bound = (b1 + b2) * 1.001f + (res_sc ? res_sc[2] : 0.f);
  if (!isfinite(bound)) bound = 3.0e38f;
  float s = 1.f;
  if (bound > 0.f) {
    int e;
    frexpf(bound, &e);                         // bound = f * 2^e, f in [0.5, 1)
    int k = 15 - e;
    k = k < -100 ? -100 : (k > 100 ? 100 : k);
    s = ldexpf(1.f, k);
  }
  sc[0] = s;
  sc[1] = 1.f / s;
  sc[2] = bound;
  sc[3] = 0.f;
}

__global__ void __launch_bounds__(1024)
act_scale_kernel(const double* __restrict__ stats, const float* __restrict__ scale,
                 const float* __restrict__ shift, double M, int C,
                 const double* __restrict__ stats2, const float* __restrict__ scale2,
                 const float* __restrict__ shift2, const float* __restrict__ res_sc,
                 float* __restrict__ sc) {
  float b1 = group_bound(stats, scale, shift, M, C);
  float b2 = stats2 ? group_bound(stats2, scale2, shift2, M, C) : 0.f;
  b1 = warp_max(b1);
  b2 = warp_max(b2);
  __shared__ float sm[2][32];
  if ((threadIdx.x & 31) == 0) { sm[0][threadIdx.x >> 5] = b1; sm[1][threadIdx.x >> 5] = b2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { b1 = fmaxf(b1, sm[0][w]); b2 = fmaxf(b2, sm[1][w]); }
    publish_act_scale(b1, b2, res_sc, sc);
  }
}

// BatchNorm finalize (as bn.cu bn_finalize_kernel) + epb_act_scale of the same layer in ONE single-CTA
// launch: group 1 is the layer being finalised, group 2 (optional) an already finalised one.
__global__ void __launch_bounds__(1024)
bn_finalize_scale_kernel(const double* __restrict__ stats, double M, int C,
                         const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                         float momentum, float* __restrict__ running_mean,
                         float* __restrict__ running_var, float* __restrict__ scale,
                         float* __restrict__ shift, float* __restrict__ mean_out,
                         float* __restrict__ invstd_out, const double* __restrict__ stats2,
                         const float* __restrict__ scale2, const float* __restrict__ shift2,
                         const float* __restrict__ res_sc, float* __restrict__ sc) {
  float b1 = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const double mean = stats[c] / M;
    double var = stats[C + c] / M - mean * mean;   // biased (normalisation)
    if (var < 0) var = 0;
    const double invstd = 1.0 / sqrt(var + (double)eps);
    const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    const float scf = (float)(g * invstd), shf = (float)(b - mean * g * invstd);
    scale[c] = scf;
    shift[c] = shf;
    if (mean_out) mean_out[c] = (float)mean;
    if (invstd_out) invstd_out[c] = (float)invstd;
    if (running_mean) {
      const double unbiased = var * (M / (M > 1.0 ? (M - 1.0) : 1.0));
      running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * mean);
      running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unbiased);
    }
    b1 = fmaxf(b1, (float)(fabs((double)scf * mean + (double)shf) + fabs((double)scf) * sqrt(M * var)));
  }
  float b2 = stats2 ? group_bound(stats2, scale2, shift2, M, C) : 0.f;
  b1 = warp_max(b1);
  b2 = warp_max(b2);
  __shared__ float sm[2][32];
  if ((threadIdx.x & 31) == 0) { sm[0][threadIdx.x >> 5] = b1; sm[1][threadIdx.x >> 5] = b2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { b1 = fmaxf(b1, sm[0][w]); b2 = fmaxf(b2, sm[1][w]); }
    publish_act_scale(b1, b2, res_sc, sc);
  }
}

// ------------------------------------------------------------------ soft-argmax backward -> split logit gradient
// dlogit = p * (s - sbar) (softargmax.cu softargmax_bwd_nhwc) written straight as the split operand of the
// final layer's backward, plus per-CTA column sums for the bias gradient (summed in a fixed order).
// Scale from a hard bound: p <= 1/sum(e^{v-m}) = lse[1], |s - sbar| <= |gx| + |gy| + |gz|.
__global__ void __launch_bounds__(1024)
softargmax_bwd_bound_kernel(const float* __restrict__ lse, const float* __restrict__ dcoords, int NJ,
                            float* __restrict__ sc) {
  float b = 0.f;
  for (int i = threadIdx.x; i < NJ; i += blockDim.x)
    b = fmaxf(b, lse[i * 2 + 1] * (fabsf(dcoords[i * 3]) + fabsf(dcoords[i * 3 + 1]) + fabsf(dcoords[i * 3 + 2])));
  b = warp_max(b);
  __shared__ float sm[32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = b;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) b = fmaxf(b, sm[w]);
    const float s = pow2_scale(b);
    sc[0] = s;
    sc[1] = 1.f / s;
  }
}

// grid (S, N), block C4 * ppi (C4 = J*D/4 channel quads, ppi pixels per trip); as softargmax_bwd_nhwc
__global__ void softargmax_bwd_split_kernel(const float* __restrict__ logits, int J, int D, int H, int W,
                                            int S, int ppi, const float* __restrict__ coords,
                                            const float* __restrict__ lse,
                                            const float* __restrict__ dcoords,
                                            const float* __restrict__ sc, uint2* __restrict__ planes,
                                            int64_t total4, float* __restrict__ parts, int nplanes) {
  extern __shared__ float4 shq[];            // [blockDim]
  const int n = blockIdx.y, sp = blockIdx.x;
  const int C4 = (J * D) >> 2;
  const int HW = H * W;
  const int per = (HW + S - 1) / S;
  const int pbeg = sp * per, pend = min(HW, pbeg + per);
  const int c4 = threadIdx.x % C4, sub = threadIdx.x / C4;
  const int D4 = D >> 2;
  const int j = c4 / D4;
  const float z0 = (float)((c4 % D4) << 2);
  const int nj = n * J + j;
  const float m = lse[nj * 2], inv = lse[nj * 2 + 1];
  const float gx = dcoords[nj * 3] / W, gy = dcoords[nj * 3 + 1] / H, gz = dcoords[nj * 3 + 2] / D;
  const float sbar = gx * (coords[nj * 3] + 0.5f) * W + gy * (coords[nj * 3 + 1] + 0.5f) * H +
                     gz * (coords[nj * 3 + 2] + 0.5f) * D;
  const float s = sc[0];
  const int64_t img = (int64_t)n * HW * C4 + c4;
  const float4* base = reinterpret_cast<const float4*>(logits) + img;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int pix = pbeg + sub;
  int y = pix / W, x = pix - y * W;
  for (; pix < pend; pix += ppi) {
    const float4 v = ldg_stream(base + (int64_t)pix * C4);
    const float s0 = gx * x + gy * y + gz * z0 - sbar;
    float4 o;
    o.x = __expf(v.x - m) * inv * (s0);
    o.y = __expf(v.y - m) * inv * (s0 + gz);
    o.z = __expf(v.z - m) * inv * (s0 + 2.f * gz);
    o.w = __expf(v.w - m) * inv * (s0 + 3.f * gz);
    uint2 hi, lo;
    split2(o.x, o.y, s, hi.x, lo.x);
    split2(o.z, o.w, s, hi.y, lo.y);
    const int64_t i = img + (int64_t)pix * C4;
    planes[i] = hi;
    if (nplanes == 2) planes[total4 + i] = lo;
    acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
    x += ppi;
    while (x >= W) { x -= W; ++y; }
  }
  shq[threadIdx.x] = acc;
  __syncthreads();
  if (sub == 0) {
    for (int q = 1; q < ppi; ++q) {
      const float4 t = shq[q * C4 + c4];
      acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
    }
    reinterpret_cast<float4*>(parts)[((int64_t)n * S + sp) * C4 + c4] = acc;
  }
}

// out[c] = sum over rows of parts[r][c] in a fixed order (8 channels x 32 row groups per CTA)
__global__ void __launch_bounds__(256)
colsum_parts_kernel(const float* __restrict__ parts, int rows, int C, float* __restrict__ out) {
  const int ch = threadIdx.x & 7, g = threadIdx.x >> 3;
  const int c = blockIdx.x * 8 + ch;
  double a = 0;
  if (c < C) {
    for (int r0 = g; r0 < rows; r0 += 32 * 16) {     // 16 independent loads in flight
      float v[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int r = r0 + 32 * u;
        v[u] = (r < rows) ? __ldg(parts + (int64_t)r * C + c) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) a += (double)v[u];
    }
  }
  __shared__ double sa[32][8];
  sa[g][ch] = a;
  __syncthreads();
#pragma unroll
  for (int half = 16; half > 0; half >>= 1) {
    if (g < half) sa[g][ch] += sa[g + half][ch];
    __syncthreads();
  }
  if (g == 0 && c < C) out[c] = (float)sa[0][ch];
}

__global__ void avgpool_split_kernel(const __half* __restrict__ x, const float* __restrict__ x_sc,
                                     float* __restrict__ y, int N, int HW, int C, int planes) {
  const int n = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const int64_t plane = (int64_t)N * HW * C;
  float acc = 0.f;
  for (int p = 0; p < HW; ++p) {
    const int64_t i = ((int64_t)n * HW + p) * C + c;
    acc += planes == 2 ? __half2float(x[i]) + __half2float(x[plane + i]) : __half2float(x[i]);
  }
  y[(int64_t)n * C + c] = acc * x_sc[1] / (float)HW;
}

}  // namespace

#define EPB_API extern "C" __attribute__((visibility("default")))

EPB_API int epb_bn_act_split(const float* x, const float* scale, const float* shift, const float* r,
                             const float* rscale, const float* rshift, const epb_half* r_split,
                             const float* r_sc, int relu, int64_t M, int C, epb_half* y,
                             const float* y_sc, uint8_t* mask_bits, int planes, epb_stream_t stream) {
  EPB_CHECK_ARG(x && y && y_sc && M > 0 && C > 0 && C % 8 == 0);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  EPB_CHECK_ARG((scale == nullptr) == (shift == nullptr));
  EPB_CHECK_ARG((rscale == nullptr) == (rshift == nullptr));
  EPB_CHECK_ARG(!(r && r_split) && ((r_split == nullptr) == (r_sc == nullptr)));
  EPB_CHECK_ARG(!rscale || r);
  const int64_t total8 = M * (C / 8);
  bn_act_split_kernel<<<ew_blocks(total8), kThreads, 0, as_stream(stream)>>>(
      x, scale, shift, r, rscale, rshift, reinterpret_cast<const uint4*>(r_split), r_sc, relu, total8,
      C / 8, reinterpret_cast<uint4*>(y), y_sc, mask_bits, planes);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_bn_relu_maxpool_split(const float* x, const float* scale, const float* shift,
                                      epb_half* y, const float* y_sc, uint8_t* argidx, int N, int H,
                                      int W, int C, int planes, epb_stream_t stream) {
  EPB_CHECK_ARG(x && scale && shift && y && y_sc && N > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  const int Ho = (H + 2 - 3) / 2 + 1, Wo = (W + 2 - 3) / 2 + 1;
  const int64_t total = (int64_t)N * Ho * Wo * (C / 8);
  bn_relu_maxpool_split_kernel<<<ew_blocks(total), kThreads, 0, as_stream(stream)>>>(
      x, scale, shift, reinterpret_cast<uint4*>(y), y_sc, reinterpret_cast<uint2*>(argidx), N, H, W,
      C / 8, planes);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_im2col_split(const float* img_nchw, epb_half* col, const float* col_sc, int N, int C,
                             int Hi, int Wi, int kh, int kw, int stride, int pad, int Ho, int Wo,
                             int Kpad, int planes, epb_stream_t stream) {
  EPB_CHECK_ARG(img_nchw && col && col_sc && N > 0 && C > 0 && Kpad % 8 == 0 && Kpad >= kh * kw * C);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  const int64_t total = (int64_t)N * Ho * Wo * (Kpad / 8);
  EPB_CHECK_ARG(Kpad <= 4096);
  {
    const int tw = stride * (kSeg - 1) + kw, segs = (Wo + kSeg - 1) / kSeg;
    const size_t smem = ((size_t)Kpad + (size_t)C * kh * tw) * sizeof(int);
    const int64_t ctas = (int64_t)N * Ho * segs;
    if (smem <= 48 * 1024 && ctas < (1LL << 31)) {
      im2col_split_tiled_kernel<<<(unsigned)ctas, kThreads, smem, as_stream(stream)>>>(
          img_nchw, reinterpret_cast<uint4*>(col), col_sc, N, C, Hi, Wi, kh, kw, stride, pad, Ho, Wo, Kpad,
          segs, tw, planes);
      EPB_LAUNCH_CHECK();
      return EPB_OK;
    }
  }
  im2col_split_kernel<<<ew_blocks(total), kThreads, 2 * Kpad * sizeof(int), as_stream(stream)>>>(
      img_nchw, reinterpret_cast<uint4*>(col), col_sc, N, C, Hi, Wi, kh, kw, stride, pad, Ho, Wo, Kpad,
      planes);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_split16_batch(const epb_split_job* jobs, int njobs, long long total_blocks,
                              uint32_t* amax_ws, int planes, epb_stream_t stream) {
  EPB_CHECK_ARG(jobs && amax_ws && njobs > 0 && total_blocks > 0 && total_blocks < (1LL << 31));
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  cudaStream_t st = as_stream(stream);
  EPB_CUDA(cudaMemsetAsync(amax_ws, 0, sizeof(uint32_t) * njobs, st));
  split_amax_kernel<<<(unsigned)total_blocks, kThreads, 0, st>>>(jobs, njobs, amax_ws);
  EPB_LAUNCH_CHECK();
  split_apply_kernel<<<(unsigned)total_blocks, kThreads, 0, st>>>(jobs, njobs, amax_ws, planes);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

// launch geometry of the partial pass: the three resident CTAs per SM, >= 4 rows per thread
static int bn_bwd_workers(const RowMap& rm, int64_t M) {
  const int64_t nblk = (M + rm.rpi - 1) / rm.rpi;
  int64_t workers = (nblk + 3) / 4;
  const int64_t cap = (int64_t)kNumSMs * 3 / rm.chunks > 1 ? (int64_t)kNumSMs * 3 / rm.chunks : 1;
  if (workers > cap) workers = cap;
  return (int)(workers < 1 ? 1 : workers);
}
// scratch of this (device, stream): parts[4][W][C] | coef[2C] | bound
static int bn_bwd_scratch(int W, int C, cudaStream_t st, float** parts, float** coef, uint32_t** bound) {
  void* p = nullptr;
  const size_t nparts = (size_t)4 * W * C;
  size_t bytes = (nparts + 2 * (size_t)C + 4) * sizeof(float);
  const size_t usual = ((size_t)4 * 3 * kNumSMs * 2048 + 2 * 2048 + 4) * sizeof(float);   // every ResNet layer
  if (bytes < usual) bytes = usual;
  int rc = epb_workspace(EPB_WS_BNPART, bytes, st, &p);
  if (rc) return rc;
  *parts = static_cast<float*>(p);
  *coef = *parts + nparts;
  *bound = reinterpret_cast<uint32_t*>(*coef + 2 * (size_t)C);
  return EPB_OK;
}

static void launch_bn_bwd_partial(const float* dy, const float* x, const epb_half* mask_hi,
                                  const float* scale, const float* shift, const float* mean,
                                  const float* invstd, int relu, int64_t M, int C, const RowMap& rm,
                                  int W, float* parts, uint32_t* bound, cudaStream_t st,
                                  int mask_kind = 1) {
  auto k = mask_kind == 2 ? bn_bwd_partial_kernel<2> : (mask_hi ? bn_bwd_partial_kernel<1> : bn_bwd_partial_kernel<0>);
  k<<<dim3(W, rm.chunks), kThreads, 0, st>>>(
      reinterpret_cast<const float4*>(dy), reinterpret_cast<const float4*>(x),
      reinterpret_cast<const uint2*>(mask_hi), reinterpret_cast<const float4*>(scale),
      reinterpret_cast<const float4*>(shift), reinterpret_cast<const float4*>(mean),
      reinterpret_cast<const float4*>(invstd), relu, M, C, rm, parts, bound);
}

EPB_API int epb_bn_bwd_reduce_mx(const float* dy, const float* x, const epb_half* mask_hi,
                                 const float* scale, const float* shift, const float* mean,
                                 const float* invstd, int relu, int64_t M, int C, double* sums,
                                 float* maxes, epb_stream_t stream) {
  EPB_CHECK_ARG(dy && x && scale && shift && mean && invstd && sums && maxes);
  EPB_CHECK_ARG(M > 0 && C > 0 && C % 4 == 0);
  cudaStream_t st = as_stream(stream);
  const RowMap rm = make_rowmap(C);
  const int W = bn_bwd_workers(rm, M);
  float *parts, *coef;
  uint32_t* bound;
  int rc = bn_bwd_scratch(W, C, st, &parts, &coef, &bound);
  if (rc) return rc;
  launch_bn_bwd_partial(dy, x, mask_hi, scale, shift, mean, invstd, relu, M, C, rm, W, parts, nullptr, st);
  EPB_LAUNCH_CHECK();
  bn_bwd_combine_kernel<<<(C + 7) / 8, 256, 0, st>>>(parts, W, (double)M, C, sums, maxes, nullptr,
                                                        nullptr, nullptr, nullptr, nullptr, nullptr);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_bn_bwd_split(const float* dy, const float* x, const epb_half* mask_hi,
                             const uint8_t* mask_bits, const float* scale, const float* shift, const float* mean,
                             const float* invstd, const float* gamma, int relu, int64_t M, int C,
                             epb_half* dz, float* dz_sc, float* dy_masked, float* dgamma,
                             float* dbeta, int planes, epb_stream_t stream) {
  EPB_CHECK_ARG(dy && x && scale && shift && mean && invstd && dz && dz_sc);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  EPB_CHECK_ARG(M > 0 && C > 0 && C % 4 == 0);
  EPB_CHECK_ARG(!(mask_hi && mask_bits) && (!mask_bits || C % 8 == 0));
  const int mask_kind = mask_bits ? 2 : 1;
  if (mask_bits) mask_hi = reinterpret_cast<const epb_half*>(mask_bits);     // one pointer, kind says how to read it
  cudaStream_t st = as_stream(stream);
  const RowMap rm = make_rowmap(C);
  const int W = bn_bwd_workers(rm, M);
  float *parts, *coef;
  uint32_t* bound;
  int rc = bn_bwd_scratch(W, C, st, &parts, &coef, &bound);
  if (rc) return rc;
  launch_bn_bwd_partial(dy, x, mask_hi, scale, shift, mean, invstd, relu, M, C, rm, W, parts, bound, st,
                        mask_kind);
  EPB_LAUNCH_CHECK();
  bn_bwd_combine_kernel<<<(C + 7) / 8, 256, 0, st>>>(parts, W, (double)M, C, nullptr, nullptr, coef,
                                                        gamma, invstd, dgamma, dbeta, bound);
  EPB_LAUNCH_CHECK();
  const int64_t total4 = M * (C / 4);
  bn_bwd_apply_split_kernel<<<ew_blocks(total4), kThreads, 0, st>>>(
      reinterpret_cast<const float4*>(dy), reinterpret_cast<const float4*>(x),
      reinterpret_cast<const uint2*>(mask_hi), reinterpret_cast<const float4*>(scale),
      reinterpret_cast<const float4*>(shift), reinterpret_cast<const float4*>(mean),
      reinterpret_cast<const float4*>(invstd), reinterpret_cast<const float4*>(gamma), relu,
      reinterpret_cast<const float4*>(coef), reinterpret_cast<const float4*>(coef + C),
      reinterpret_cast<uint2*>(dz), dz_sc, reinterpret_cast<const float*>(bound),
      reinterpret_cast<float4*>(dy_masked), total4, C / 4, mask_kind == 2, planes);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_bn_bwd_apply_split(const float* dy, const float* x, const epb_half* mask_hi,
                                   const float* scale, const float* shift, const float* mean,
                                   const float* invstd, const float* gamma, int relu,
                                   const double* sums, const float* maxes, int64_t M, int C,
                                   epb_half* dz, float* dz_sc, float* dy_masked, float* dgamma,
                                   float* dbeta, int planes, epb_stream_t stream) {
  EPB_CHECK_ARG(dy && x && scale && shift && mean && invstd && sums && maxes && dz && dz_sc);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  EPB_CHECK_ARG(M > 0 && C > 0 && C % 4 == 0);
  cudaStream_t st = as_stream(stream);
  float* mx = const_cast<float*>(maxes);      // consumed here: overwritten by the coefficients
  bn_bwd_coef_split_kernel<<<1, 1024, 0, st>>>(sums, mx, (double)M, C, gamma, invstd, dz_sc, dgamma,
                                               dbeta);
  EPB_LAUNCH_CHECK();
  const int64_t total4 = M * (C / 4);
  bn_bwd_apply_split_kernel<<<ew_blocks(total4), kThreads, 0, st>>>(
      reinterpret_cast<const float4*>(dy), reinterpret_cast<const float4*>(x),
      reinterpret_cast<const uint2*>(mask_hi), reinterpret_cast<const float4*>(scale),
      reinterpret_cast<const float4*>(shift), reinterpret_cast<const float4*>(mean),
      reinterpret_cast<const float4*>(invstd), reinterpret_cast<const float4*>(gamma), relu,
      reinterpret_cast<const float4*>(mx), reinterpret_cast<const float4*>(mx + C),
      reinterpret_cast<uint2*>(dz), dz_sc, nullptr, reinterpret_cast<float4*>(dy_masked), total4, C / 4, 0,
      planes);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_avgpool_split(const epb_half* x, const float* x_sc, float* y, int N, int HW, int C,
                              int planes, epb_stream_t stream) {
  EPB_CHECK_ARG(x && x_sc && y && N > 0 && HW > 0 && C > 0);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  avgpool_split_kernel<<<dim3((C + 127) / 128, N), 128, 0, as_stream(stream)>>>(
      reinterpret_cast<const __half*>(x), x_sc, y, N, HW, C, planes);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_act_scale(const double* stats, const float* scale, const float* shift, int64_t M,
                          int C, const double* stats2, const float* scale2, const float* shift2,
                          const float* res_sc, float* sc, epb_stream_t stream) {
  EPB_CHECK_ARG(stats && scale && shift && sc && M > 0 && C > 0);
  EPB_CHECK_ARG((stats2 == nullptr) == (scale2 == nullptr) && (scale2 == nullptr) == (shift2 == nullptr));
  act_scale_kernel<<<1, 1024, 0, as_stream(stream)>>>(stats, scale, shift, (double)M, C, stats2,
                                                      scale2, shift2, res_sc, sc);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_bn_finalize_scale(const double* stats, int64_t M, int C, const float* gamma,
                                  const float* beta, float eps, float momentum, float* running_mean,
                                  float* running_var, float* scale, float* shift, float* mean,
                                  float* invstd, const double* stats2, const float* scale2,
                                  const float* shift2, const float* res_sc, float* sc,
                                  epb_stream_t stream) {
  EPB_CHECK_ARG(stats && scale && shift && sc && M > 0 && C > 0);
  EPB_CHECK_ARG((running_mean == nullptr) == (running_var == nullptr));
  EPB_CHECK_ARG((stats2 == nullptr) == (scale2 == nullptr) && (scale2 == nullptr) == (shift2 == nullptr));
  bn_finalize_scale_kernel<<<1, 1024, 0, as_stream(stream)>>>(
      stats, (double)M, C, gamma, beta, eps, momentum, running_mean, running_var, scale, shift, mean,
      invstd, stats2, scale2, shift2, res_sc, sc);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

EPB_API int epb_softargmax_bwd_split(const float* logits, int N, int J, int D, int H, int W,
                                     const float* coords, const float* lse_ws, const float* dcoords,
                                     epb_half* dlogits16, float* sc, float* dbias, int planes,
                                     epb_stream_t stream) {
  EPB_CHECK_ARG(logits && coords && lse_ws && dcoords && dlogits16 && sc);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  EPB_CHECK_ARG(N > 0 && J > 0 && D > 0 && H > 0 && W > 0 && D % 4 == 0);
  const int C4 = J * D / 4;
  EPB_CHECK_ARG(C4 <= 1024);
  cudaStream_t st = as_stream(stream);
  const int ppi = (512 / C4) > 0 ? (512 / C4) : 1;
  int S = 1;
  while (N * S < 8 * kNumSMs && (H * W) / (S * 2) >= 16 * ppi) S *= 2;
  void* parts = nullptr;
  int rc = epb_workspace(EPB_WS_SABWD, (size_t)N * S * C4 * 4 * sizeof(float), st, &parts);
  if (rc) return rc;
  softargmax_bwd_bound_kernel<<<1, 1024, 0, st>>>(lse_ws, dcoords, N * J, sc);
  EPB_LAUNCH_CHECK();
  const int threads = C4 * ppi;
  softargmax_bwd_split_kernel<<<dim3(S, N), threads, threads * sizeof(float4), st>>>(
      logits, J, D, H, W, S, ppi, coords, lse_ws, dcoords, sc, reinterpret_cast<uint2*>(dlogits16),
      (int64_t)N * H * W * C4, static_cast<float*>(parts), planes);
  EPB_LAUNCH_CHECK();
  if (dbias) {
    colsum_parts_kernel<<<(C4 * 4 + 7) / 8, 256, 0, st>>>(static_cast<const float*>(parts), N * S,
                                                            C4 * 4, dbias);
    EPB_LAUNCH_CHECK();
  }
  return EPB_OK;
}

EPB_API int epb_split16(const float* src, long long n, epb_half* dst, float* sc, uint32_t* amax_ws,
                        int planes, epb_stream_t stream) {
  EPB_CHECK_ARG(src && dst && sc && amax_ws && n > 0 && n % 4 == 0);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  cudaStream_t st = as_stream(stream);
  EPB_CUDA(cudaMemsetAsync(amax_ws, 0, sizeof(uint32_t), st));
  const int64_t n4 = n / 4;
  split_amax_one_kernel<<<ew_blocks(n4), kThreads, 0, st>>>(reinterpret_cast<const float4*>(src), n4,
                                                            amax_ws);
  EPB_LAUNCH_CHECK();
  split_apply_one_kernel<<<ew_blocks(n4), kThreads, 0, st>>>(reinterpret_cast<const float4*>(src), n4,
                                                             amax_ws, reinterpret_cast<uint2*>(dst), sc, planes);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}
