// Split-fp16 ("f16x3") weight-gradient kernel of the tap-list implicit GEMM (include/epb.h,
// epb_conv16_wgrad; cuDNN wgrad behind the autograd of lib/models/pose3d_resnet.py:12-15,
// 55-60,99,116-122,171-178):
//
//   dw[co][wt[t]][ci] += (1 / (s_in * s_dout)) * sum_m in[pix_in(m, t)][ci] * dout[pix_out(m)][co]
//
// GEMM view: D[(t, ci), co] with the reduction over phase-grid pixels m.  Both operands are
// MN-major for the tensor core (channels contiguous in NHWC memory, the reduction index
// strides over pixel rows) and come straight from the fp16 planes by TMA: a tile of 64 pixels
// x 64 channels is one 5-D box load -- 64 rows of 128 bytes, exactly the SWIZZLE_128B MN-major
// atom sequence tcgen05 reads (8-row atoms 1024 B apart, 64-channel chunks LBO apart).
// The M side is a list of CHUNKS (tap, 64-channel block): 4 chunks per CTA pair (M = 256,
// tcgen05 cta_group::2), each chunk its own tap-shifted box, so every tap of a 64-channel
// layer still fills the M rows; the N side is min(Cout, 256) output channels, half per CTA.
// The pixel range is split across clusters; partial tiles go to `ws` and are summed in split
// order by a second kernel (deterministic; no atomics).
// Template NP = 1 is the single-pass ("f16") form: hi planes only, one tcgen05.mma per k-step,
// a deeper ring in the smem the lo boxes no longer take.
#include "split16_common.cuh"

namespace {

constexpr int KT = 64;                 // pixels per stage (4 MMAs of K = 16)
constexpr int kThreadsW16 = 192;
constexpr int kChunk = KT * 128;       // bytes of one (64 pixels x 64 channels) box

struct PlanW16 {
  int N, Hp, Wp;
  int Cin, Cout, Tw;
  int T, CB, CH;                 // taps, 64-channel blocks per tap, chunks = T * CB
  int tw, th, tn, tiles_w, tiles_h, ptiles;
  int groups, n_tiles, splits, tiles_per_split;
  int swap;                      // 1: M side = 64-channel blocks of dout, N side = input channels
  int Nn;                        // channels on the N side (Cout, or Cin when swapped)
  int bdw, bdh;                  // box offset of the N-side operand (the tap, when swapped)
  int wt[EPB_MAX_TAPS];
  short dwq[EPB_MAX_TAPS], dhq[EPB_MAX_TAPS];
  unsigned char map[EPB_MAX_TAPS];
};

struct MapsW16 {
  CUtensorMap a[4];
  CUtensorMap d;
};

// NP: operand planes (2: hi + lo, three passes; 1: hi only, one pass)
template <int BN, int NP>
struct CfgW16 {
  static constexpr int BCH = BN / 128;                   // 64-channel chunks of dout per CTA
  static constexpr int A_PLANE = 2 * kChunk;
  static constexpr int B_PLANE = BCH * kChunk;
  static constexpr int STAGE = NP * A_PLANE + NP * B_PLANE;
  // two planes: the measured ring (<= 6 stages in 192 KB); one plane: as deep as the 227 KB
  // allow, up to the 8 full / empty barrier pairs (BN 256: 7, BN 128: 8 stages)
  static constexpr int S_ = NP == 2 ? (192 * 1024) / STAGE : (227 * 1024 - 1024 - 256) / STAGE;
  static constexpr int S_MAX = NP == 2 ? 6 : 8;
  static constexpr int S = S_ > S_MAX ? S_MAX : S_;
  static constexpr int SMEM = S * STAGE + 1024 + 256;
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
};

template <int BN, int NP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsW16, 1)
wgrad16_kernel(const __grid_constant__ PlanW16 P, const __grid_constant__ MapsW16 maps,
               const float* __restrict__ in_sc, const float* __restrict__ dout_sc,
               float* __restrict__ dw, float* __restrict__ ws) {
  using C = CfgW16<BN, NP>;
  const int crank = (int)tc::cluster_ctarank();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = tc::smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);
  uint8_t* ctrl = sm + C::S * C::STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ctrl);          // full[8], empty[8], done
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(ctrl + 8 * 17);
  const uint32_t bar0 = tc::smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (8 + s); };
  const uint32_t done_bar = bar0 + 8u * 16;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // work item: cluster id = ((split * n_tiles + nt) * groups + grp)
  int wi = (int)tc::cluster_id_x();
  const int grp = wi % P.groups; wi /= P.groups;
  const int nt = wi % P.n_tiles;
  const int split = wi / P.n_tiles;
  const int pt0 = split * P.tiles_per_split;
  const int pt1 = min(P.ptiles, pt0 + P.tiles_per_split);
  const int nst = pt1 - pt0;                                   // stages of this cluster (>= 1)

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::S; ++s) {
      tc::mbar_init(full_bar(s), 1);
      tc::mbar_init(empty_bar(s), 1);
    }
    tc::mbar_init(done_bar, 1);
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc_pair<BN>(tc::smem_u32(tmem_ptr));
  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =================================================== TMA producer
    if (lane == 0) {
      for (int v = 0; v < 4; ++v) tc::tma_prefetch_desc(&maps.a[v]);
      tc::tma_prefetch_desc(&maps.d);
      // this CTA's two chunks (clamped: rows of a chunk past the end are computed, never stored)
      int ct[2], cc[2];
      for (int j = 0; j < 2; ++j) {
        const int c = min(grp * 4 + crank * 2 + j, P.CH - 1);
        ct[j] = c / P.CB;
        cc[j] = (c % P.CB) * 64;
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int pt = pt0; pt < pt1; ++pt) {
        int it = pt;
        const int w0 = (it % P.tiles_w) * P.tw; it /= P.tiles_w;
        const int h0 = (it % P.tiles_h) * P.th;
        const int n0 = (it / P.tiles_h) * P.tn;
        tc::mbar_wait(empty_bar(stage), phase ^ 1);
        if (crank == 0) tc::mbar_arrive_expect_tx(full_bar(stage), 2 * C::STAGE);
        const uint32_t lead_bar = tc::mapa(full_bar(stage), 0);
        const uint32_t a_dst = base + stage * C::STAGE;
        const uint32_t b_dst = a_dst + NP * C::A_PLANE;
#pragma unroll
        for (int pl = 0; pl < NP; ++pl) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int t = ct[j];
            tc::tma_load_5d_pair(a_dst + pl * C::A_PLANE + j * kChunk, &maps.a[P.map[t]], lead_bar,
                                 cc[j], w0 + P.dwq[t], h0 + P.dhq[t], n0, pl);
          }
#pragma unroll
          for (int jb = 0; jb < C::BCH; ++jb)
            tc::tma_load_5d_pair(b_dst + pl * C::B_PLANE + jb * kChunk, &maps.d, lead_bar,
                                 nt * BN + (crank * C::BCH + jb) * 64, w0 + P.bdw, h0 + P.bdh, n0, pl);
        }
        if (++stage == C::S) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // =================================================== MMA issuer (leader CTA)
    if (lane == 0 && crank == 0) {
      constexpr uint32_t idesc = tc::idesc_f16(256, BN, 1, 1);        // both operands MN-major
      int stage = 0;
      uint32_t phase = 0;
      for (int k = 0; k < nst; ++k) {
        tc::mbar_wait_cluster(full_bar(stage), phase);
        tc::tc_fence_after();
        const uint32_t a_hi = base + stage * C::STAGE;
        const uint32_t b_hi = a_hi + NP * C::A_PLANE;
#pragma unroll
        for (int ks = 0; ks < KT / 16; ++ks) {
          const uint64_t ah = tc::desc_mnmajor16_sw128(a_hi + ks * 2048, kChunk, 1024);
          const uint64_t bh = tc::desc_mnmajor16_sw128(b_hi + ks * 2048, kChunk, 1024);
          if (NP == 2) {
            const uint64_t al = tc::desc_mnmajor16_sw128(a_hi + C::A_PLANE + ks * 2048, kChunk, 1024);
            const uint64_t bl = tc::desc_mnmajor16_sw128(b_hi + C::B_PLANE + ks * 2048, kChunk, 1024);
            tc::mma_f16_pair(tmem_base, al, bh, idesc, (k | ks) != 0);
            tc::mma_f16_pair(tmem_base, ah, bl, idesc, 1);
            tc::mma_f16_pair(tmem_base, ah, bh, idesc, 1);
          } else {
            tc::mma_f16_pair(tmem_base, ah, bh, idesc, (k | ks) != 0);
          }
        }
        tc::mma_commit_pair(empty_bar(stage));
        if (++stage == C::S) { stage = 0; phase ^= 1; }
      }
      tc::mma_commit_pair(done_bar);
    }
  } else {
    // =================================================== epilogue (4 warps, own TMEM lanes)
    const int q = warp & 3;
    const int c = grp * 4 + crank * 2 + (q >> 1);             // chunk of this warp's 32 rows
    tc::mbar_wait(done_bar, 0);
    tc::tc_fence_after();
    if (c < P.CH) {
      const int64_t K = (int64_t)P.Tw * P.Cin;
      const float alpha = in_sc[1] * dout_sc[1];
      float* dst = P.splits > 1 ? ws + (int64_t)split * P.Cout * K : dw;
      const int rowc = (q & 1) * 32 + lane;                   // this lane's row inside the chunk
      // normal : row = input channel ci of tap t,  column = output channel co
      // swapped: row = output channel co,          column = input channel ci (T == 1)
      const int t = P.swap ? 0 : c / P.CB;
      const int64_t row_off = P.swap ? (int64_t)(c * 64 + rowc) * K + (int64_t)P.wt[0] * P.Cin
                                     : (int64_t)P.wt[t] * P.Cin + (c % P.CB) * 64 + rowc;
      const int64_t col_stride = P.swap ? 1 : K;
#pragma unroll 1
      for (int chunk = 0; chunk < BN / 32; ++chunk) {
        const int col0 = nt * BN + chunk * 32;
        if (col0 >= P.Nn) break;
        uint32_t rg[32];
        tc::tmem_ld32(tmem_base + chunk * 32 + ((uint32_t)(q * 32) << 16), rg);
        tc::tmem_ld_wait();
        if (P.splits > 1) {
#pragma unroll
          for (int cc = 0; cc < 32; ++cc)
            if (col0 + cc < P.Nn) dst[row_off + (int64_t)(col0 + cc) * col_stride] = __uint_as_float(rg[cc]);
        } else {
#pragma unroll
          for (int cc = 0; cc < 32; ++cc)
            if (col0 + cc < P.Nn) {
              float* o = dst + row_off + (int64_t)(col0 + cc) * col_stride;
              *o += alpha * __uint_as_float(rg[cc]);
            }
        }
      }
    }
  }

  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();
  if (warp == 1) {
    tc::tc_fence_after();
    tc::tmem_dealloc_pair<BN>(tmem_base);
  }
}

// dw[co][wt[t]][ci] += alpha * sum_s ws[s][co][wt[t]][ci]   (fixed order)
__global__ void __launch_bounds__(256)
wgrad16_reduce_kernel(const __grid_constant__ PlanW16 P, const float* __restrict__ in_sc,
                      const float* __restrict__ dout_sc, const float* __restrict__ ws,
                      float* __restrict__ dw) {
  const int C4 = P.Cin / 4;
  const int64_t K = (int64_t)P.Tw * P.Cin;
  const int64_t total = (int64_t)P.Cout * P.T * C4;
  const int64_t plane4 = (int64_t)P.Cout * K / 4;
  const float alpha = in_sc[1] * dout_sc[1];
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * 256) {
    const int c4 = (int)(i % C4);
    const int t = (int)((i / C4) % P.T);
    const int64_t co = i / ((int64_t)C4 * P.T);
    const int64_t o4 = (co * K + (int64_t)P.wt[t] * P.Cin) / 4 + c4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < P.splits; ++s) {
      const float4 v = reinterpret_cast<const float4*>(ws)[s * plane4 + o4];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    float4* o = reinterpret_cast<float4*>(dw) + o4;
    float4 d = *o;
    d.x += alpha * acc.x; d.y += alpha * acc.y; d.z += alpha * acc.z; d.w += alpha * acc.w;
    *o = d;
  }
}

template <int BN, int NP>
int launch_w16(const PlanW16& P, const MapsW16& maps, const float* in_sc, const float* dout_sc,
               float* dw, float* ws, cudaStream_t st) {
  using C = CfgW16<BN, NP>;
  static bool attr_set = false;
  if (!attr_set) {
    EPB_CUDA(cudaFuncSetAttribute(wgrad16_kernel<BN, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  C::SMEM));
    attr_set = true;
  }
  const int64_t clusters = (int64_t)P.groups * P.n_tiles * P.splits;
  EPB_CHECK_ARG(clusters < (1LL << 30));
  wgrad16_kernel<BN, NP><<<(unsigned)(2 * clusters), kThreadsW16, C::SMEM, st>>>(P, maps, in_sc, dout_sc,
                                                                           dw, ws);
  EPB_LAUNCH_CHECK();
  if (P.splits > 1) {
    const int64_t total = (int64_t)P.Cout * P.T * (P.Cin / 4);
    int64_t blocks = (total + 255) / 256;
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    wgrad16_reduce_kernel<<<(unsigned)blocks, 256, 0, st>>>(P, in_sc, dout_sc, ws, dw);
    EPB_LAUNCH_CHECK();
  }
  return EPB_OK;
}

}  // namespace

extern "C" __attribute__((visibility("default"))) int epb_conv16_wgrad(
    const epb_conv_geom* g, const epb_half* in, const float* in_sc, const epb_half* dout,
    const float* dout_sc, float* dw, float* ws, long long ws_floats, int planes, epb_stream_t stream) {
  int rc = epb_conv_geom_check(g);
  if (rc) return rc;
  EPB_CHECK_ARG(in && in_sc && dout && dout_sc && dw);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  EPB_CHECK_ARG(g->Cin % 64 == 0 && g->Cout % 64 == 0);
  EPB_CHECK_ARG((g->is == 1 || g->is == 2) && (g->os == 1 || g->os == 2));
  PlanW16 P;
  MapsW16 maps;
  memset(&maps, 0, sizeof(maps));
  P.Cin = g->Cin; P.Cout = g->Cout; P.Tw = g->Tw; P.T = g->T; P.CB = g->Cin / 64;
  P.CH = P.T * P.CB;
  // A 1x1 layer with few input channels leaves most of the 4 M-side chunks of a CTA pair
  // empty: put the output channels on the M side instead (D^T; same products, same sums)
  P.swap = (g->T == 1 && P.CH < 4 && g->Cout / 64 > P.CH) ? 1 : 0;
  P.bdw = P.bdh = 0;
  const bool dense = g->T == 1 && g->is == 1 && g->os == 1 && g->dh[0] == 0 && g->dw[0] == 0 &&
                     g->Hp == g->Hi && g->Wp == g->Wi && g->Hp == g->Ho && g->Wp == g->Wo;
  int N = g->N, Hi = g->Hi, Wi = g->Wi, Ho = g->Ho, Wo = g->Wo;
  P.N = g->N; P.Hp = g->Hp; P.Wp = g->Wp;
  if (dense) {
    const int64_t M = (int64_t)g->N * g->Hp * g->Wp;
    EPB_CHECK_ARG(M < (1LL << 31));
    N = 1; Hi = Ho = 1; Wi = Wo = (int)M;
    P.N = 1; P.Hp = 1; P.Wp = (int)M;
  }
  epb_choose_tile(P.N, P.Hp, P.Wp, KT, P.tw, P.th, P.tn);
  P.tiles_w = (P.Wp + P.tw - 1) / P.tw;
  P.tiles_h = (P.Hp + P.th - 1) / P.th;
  const int64_t pt = (int64_t)P.tiles_w * P.tiles_h * ((P.N + P.tn - 1) / P.tn);
  EPB_CHECK_ARG(pt < (1LL << 30));
  P.ptiles = (int)pt;
  bool need[4] = {false, false, false, false};
  for (int t = 0; t < g->T; ++t) {
    int qh, qw, dq_h, dq_w;
    epb_tap_split(g->dh[t], g->is, qh, dq_h);
    epb_tap_split(g->dw[t], g->is, qw, dq_w);
    P.map[t] = (unsigned char)(qh * 2 + qw);
    P.dhq[t] = (short)dq_h;
    P.dwq[t] = (short)dq_w;
    P.wt[t] = g->wt[t];
    need[qh * 2 + qw] = true;
  }
  CUtensorMap in_maps[4];
  memset(in_maps, 0, sizeof(in_maps));
  for (int v = 0; v < 4; ++v) {
    if (!need[v]) continue;
    rc = epb_make_act_map(&in_maps[v], in, N, Hi, Wi, g->Cin, g->is, v >> 1, v & 1, P.tw, P.th, P.tn,
                          planes);
    if (rc) return rc;
  }
  for (int v = 0; v < 4; ++v)
    if (!need[v]) {
      for (int u = 0; u < 4; ++u)
        if (need[u]) { in_maps[v] = in_maps[u]; break; }
    }
  CUtensorMap d_map;
  rc = epb_make_act_map(&d_map, dout, N, Ho, Wo, g->Cout, g->os, g->ph, g->pw, P.tw, P.th, P.tn, planes);
  if (rc) return rc;
  int bn;
  if (!P.swap) {
    for (int v = 0; v < 4; ++v) maps.a[v] = in_maps[v];
    maps.d = d_map;
    P.Nn = g->Cout;
  } else {
    // M side: the CH' = Cout / 64 blocks of dout (no tap shift); N side: the input, shifted by the tap
    for (int v = 0; v < 4; ++v) maps.a[v] = d_map;
    maps.d = in_maps[P.map[0]];
    P.bdw = P.dwq[0]; P.bdh = P.dhq[0];
    P.map[0] = 0; P.dwq[0] = 0; P.dhq[0] = 0;
    P.CB = g->Cout / 64;
    P.CH = P.CB;
    P.Nn = g->Cin;
  }
  bn = P.Nn <= 128 ? 128 : 256;
  P.n_tiles = (P.Nn + bn - 1) / bn;
  P.groups = (P.CH + 3) / 4;
  // pixel-range splits: fill one wave of cluster pairs, keep >= 8 stages per cluster, and
  // stay inside the scratch the caller gave
  const int64_t basec = (int64_t)P.groups * P.n_tiles;
  int64_t splits = (kNumSMs / 2) / basec;
  if (splits > P.ptiles / 8) splits = P.ptiles / 8;
  const int64_t per_split = (int64_t)g->Cout * g->Tw * g->Cin;
  if (!ws || splits * per_split > ws_floats) splits = ws ? ws_floats / per_split : 1;
  if (splits < 1) splits = 1;
  P.tiles_per_split = (int)((P.ptiles + splits - 1) / splits);
  P.splits = (P.ptiles + P.tiles_per_split - 1) / P.tiles_per_split;
  cudaStream_t st = as_stream(stream);
  if (planes == 1) {
    if (bn == 128) return launch_w16<128, 1>(P, maps, in_sc, dout_sc, dw, ws, st);
    return launch_w16<256, 1>(P, maps, in_sc, dout_sc, dw, ws, st);
  }
  if (bn == 128) return launch_w16<128, 2>(P, maps, in_sc, dout_sc, dw, ws, st);
  return launch_w16<256, 2>(P, maps, in_sc, dout_sc, dw, ws, st);
}
