// Host-side helpers shared by the split-fp16 tensor-core kernels (conv16.cu, wgrad16.cu):
// pixel-tile shapes and the TMA tensor maps of split activation / weight tensors.
#pragma once
#include "conv_common.cuh"
#include "tc_common.cuh"

// A tile of `rows` phase-grid pixels is the box (tw, th, tn) of the (Wp, Hp, N) grid, all
// powers of two with tw*th*tn == rows, so that ONE TMA box load brings the tile (rows in
// w-fastest order).  Chosen to minimise the covered-but-invalid pixels.
inline void epb_choose_tile(int N, int Hp, int Wp, int rows, int& tw, int& th, int& tn) {
  long long best = -1;
  tw = rows; th = 1; tn = 1;
  for (int a = rows; a >= 1; a >>= 1) {
    for (int b = rows / a; b >= 1; b >>= 1) {
      const int c = rows / (a * b);
      const long long cov = (long long)((Wp + a - 1) / a) * ((Hp + b - 1) / b) * ((N + c - 1) / c);
      if (best < 0 || cov < best) { best = cov; tw = a; th = b; tn = c; }
    }
  }
}

// 5-D map over the planes of a split NHWC tensor [planes][N][H][W][C] fp16 (planes 2: hi, lo;
// 1: hi only), viewed with spatial stride `stride` starting at pixel (qh, qw): coordinates
// (c, w', h', n, plane) address pixel (h'*stride + qh, w'*stride + qw).  Out-of-range
// coordinates (negative included) read 0.
inline int epb_make_act_map(CUtensorMap* m, const epb_half* base, int N, int H, int W, int C,
                            int stride, int qh, int qw, int tw, int th, int tn, int planes) {
  epb_encode_tiled_fn enc = epb_get_encode_tiled();
  if (!enc) {
    epb_set_error("cuTensorMapEncodeTiled entry point unavailable");
    return EPB_ECUDA;
  }
  const int Wv = (W - qw + stride - 1) / stride, Hv = (H - qh + stride - 1) / stride;
  if (Wv <= 0 || Hv <= 0) {
    epb_set_error("empty strided view");
    return EPB_EINVAL;
  }
  const cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)Wv, (cuuint64_t)Hv, (cuuint64_t)N, (cuuint64_t)planes};
  const cuuint64_t strides[4] = {(cuuint64_t)stride * C * 2, (cuuint64_t)stride * W * C * 2,
                                 (cuuint64_t)H * W * C * 2, (cuuint64_t)N * H * W * C * 2};
  const cuuint32_t box[5] = {64, (cuuint32_t)tw, (cuuint32_t)th, (cuuint32_t)tn, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  void* p = const_cast<epb_half*>(base) + ((int64_t)qh * W + qw) * C;
  CUresult cr = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, p, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    epb_set_error("cuTensorMapEncodeTiled(activation %dx%dx%dx%d stride %d box %dx%dx%d) failed (%d)",
                  N, H, W, C, stride, tw, th, tn, (int)cr);
    return EPB_ECUDA;
  }
  return EPB_OK;
}

// Tap offset d on a stride-`s` view: parity q = d mod s (non-negative), quotient (d - q) / s
inline void epb_tap_split(int d, int s, int& q, int& quot) {
  q = ((d % s) + s) % s;
  quot = (d - q) / s;
}
