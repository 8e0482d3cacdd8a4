// Split-fp16 ("f16x3") tensor-core path of the tap-list implicit GEMM (include/epb.h,
// epb_conv16_fprop): forward convs, transposed convs (one call per output phase) and both of
// their data gradients, i.e. the cuDNN call sites behind nn.Conv2d / nn.ConvTranspose2d of
// lib/models/pose3d_resnet.py:12-15,55-60,99,116-122,132,171-178 and their autograd.
//
//   out[m, co] = (1 / (s_in * s_w)) * sum_k A[m, k] * W[co, k],   m = phase-grid pixel,
//   k = (tap, ci),  A = hi + lo, W = hi + lo  (fp16 planes),
//   A*W ~= A_lo*W_hi + A_hi*W_lo + A_hi*W_hi   (three kind::f16 passes, FP32 accumulate).
// Single-pass ("f16") form, template NP = 1: the operands are the hi planes alone (10 explicit
// mantissa bits, TF32-class), A*W ~= A_hi*W_hi, one kind::f16 pass per k-step; the smem of the
// missing lo boxes deepens the operand ring.
//
// Both operands are TMA-fed: the activation planes are post-BatchNorm/ReLU (written once by
// split16.cu), so an M tile of 128 pixels is ONE 5-D box load per plane and tap -- (64 channels,
// tw, th, tn) of the (C, W, H, N, plane) tensor, shifted by the tap offset; the zero padding
// of the convolution is the TMA out-of-bounds fill, strided convs use the four parity views of
// the tensor.  Weight planes are 3-D (k, co, plane) box loads.
//
// Always CTA pairs (cluster of 2, tcgen05 cta_group::2, M = 256): each CTA holds its 128 A
// rows and HALF of the B tile's N rows, which keeps shared-memory reads under 128 B/clk at
// the kind::f16 rate.  One persistent cluster per SM pair, 6 warps per CTA:
//   warp 0    TMA producer (one lane): A hi/lo + B hi/lo boxes (hi only when NP = 1) per
//             k-block, S-deep ring;
//   warp 1    MMA issuer (leader CTA, one lane): 4 k-steps x 3 (NP = 1: 1) tcgen05.mma per k-block,
//             FP32 accumulators double buffered in TMEM;
//   warps 2-5 epilogue: tcgen05.ld -> scale / bias -> 128B-swizzled smem box -> ONE TMA store
//             (or TMA reduce-add for the accumulate form) per 32x32 block: no per-row address
//             arithmetic, rows / columns outside the tensor are clipped by the TMA unit;
//             per-channel sum / sum of squares for the following BatchNorm from the staged
//             box, accumulated in shared memory ACROSS the CTA's tiles (one atomic per column
//             and CTA instead of one per tile).
// Every mbarrier wait is bounded (trap instead of hang).
#include "split16_common.cuh"

namespace {

constexpr int BM = 128;
constexpr int kThreads16 = 192;
constexpr int kEpiWarps = 4;
constexpr int kStageBudget = 192 * 1024;

// EPB_C16_PROBE & 32: cluster 0 records clock64() at its pipeline hand-overs (epb_debug_conv16_trace):
// [role 0 producer | 1 MMA issuer | 2 epilogue warp 2 per tile | 3 epilogue warp 2 per chunk][CTA rank][256 events]
// (the per-chunk events cost instructions in the hot loop: compiled in only with -DEPB_C16_TRACE_CHUNKS)
__device__ long long g_c16_trace[4 * 2 * 256];
#define C16_TR(role, idx)                                                                      \
  do {                                                                                         \
    if (trace_on && (idx) < 256) g_c16_trace[((role) * 2 + crank) * 256 + (idx)] = clock64();   \
  } while (0)

struct Plan16 {
  int N, Hp, Wp;                 // phase grid
  int Ho, Wo, Cout, os, ph, pw;  // output tensor / phase
  int T, CB;                     // taps, channel blocks of 64 per tap
  int tw, th, tn, tiles_w, tiles_h;
  int m_tiles, n_tiles;
  int accumulate;
  int m_fastest;                 // tile order: consecutive tiles walk M (statistics runs) or N
  int probe;                     // EPB_C16_PROBE (profiling only, wrong results): 4 no stores, 8 no statistics
  int koff[EPB_MAX_TAPS];        // wt[t] * Cin: k offset of the tap inside a packed weight row
  short dwq[EPB_MAX_TAPS], dhq[EPB_MAX_TAPS];   // tap offset on its parity view
  unsigned char map[EPB_MAX_TAPS];              // parity view of the tap
};

struct Maps16 {
  CUtensorMap a[4];
  CUtensorMap w;
  CUtensorMap o;                 // fp32 output, box = 32 channels x 32 tile rows
};

// NP: operand planes (2: hi + lo, three passes; 1: hi only, one pass)
template <int BN, int NP>
struct Cfg16 {
  static constexpr int BROWS = BN / 2;                 // B rows held by this CTA
  static constexpr int A_PLANE = BM * 128;
  static constexpr int B_PLANE = BROWS * 128;
  static constexpr int A_BYTES = NP * A_PLANE;
  static constexpr int B_BYTES = NP * B_PLANE;
  static constexpr int STAGE = A_BYTES + B_BYTES;
  static constexpr int TMEM_COLS = (2 * BN <= 128) ? 128 : (2 * BN <= 256 ? 256 : 512);
  static constexpr int EPI_BYTES = kEpiWarps * 4096;           // one swizzled 32x32 fp32 box per warp
  static constexpr int STAT_BYTES = kEpiWarps * 2 * BN * 4;    // per-warp [sum | sum of squares][BN]
  static constexpr int FIXED = EPI_BYTES + 1024 /*align*/ + 1024 /*barriers*/ + STAT_BYTES;
  // two planes: the measured ring (<= 6 stages in 192 KB); one plane: as deep as the 227 KB
  // allow, up to the 8 full / empty barrier pairs (BN 256: 6, BN 128 / 64: 8 stages)
  static constexpr int S_ = NP == 2 ? kStageBudget / STAGE : (227 * 1024 - FIXED) / STAGE;
  static constexpr int S_MAX = NP == 2 ? 6 : 8;
  static constexpr int S = S_ > S_MAX ? S_MAX : S_;
  static constexpr int SMEM = S * STAGE + FIXED;
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
  static_assert(S >= 2, "ring too shallow");
};

template <int BN, int NP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads16, 1)
conv16_kernel(const __grid_constant__ Plan16 P, const __grid_constant__ Maps16 maps,
              const float* __restrict__ in_sc, const float* __restrict__ w_sc,
              const float* __restrict__ bias, float* __restrict__ out,
              double* __restrict__ stats) {
  using C = Cfg16<BN, NP>;
  const int crank = (int)tc::cluster_ctarank();
  const int tile0 = (int)tc::cluster_id_x();
  const int tstep = (int)tc::cluster_count_x();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = tc::smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);
  uint8_t* epi_stage = sm + C::S * C::STAGE;                   // [4 warps][4096], 1024-byte aligned
  uint8_t* ctrl = epi_stage + C::EPI_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ctrl);          // full[8], empty[8], tfull[2], tempty[2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(ctrl + 8 * 20);
  float* sstat = reinterpret_cast<float*>(ctrl + 1024);                      // [4 warps][2][BN]
  const uint32_t bar0 = tc::smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (8 + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (16 + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (18 + a); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool trace_on = (P.probe & 32) && tile0 == 0;
  int tr_i = 0;
#ifdef EPB_C16_TRACE_CHUNKS
  int tr_c = 0;
#endif
  const int KB = P.T * P.CB;
  const int m_pairs = (P.m_tiles + 1) / 2;
  const int total_tiles = m_pairs * P.n_tiles;
  auto nt_of = [&](int tile) { return P.m_fastest ? tile / m_pairs : tile % P.n_tiles; };
  auto mp_of = [&](int tile) { return P.m_fastest ? tile % m_pairs : tile / P.n_tiles; };

  if (threadIdx.x == 0) {
    for (int s = 0; s < C::S; ++s) {
      tc::mbar_init(full_bar(s), 1);          // the leader's arrive.expect_tx; bytes from both CTAs
      tc::mbar_init(empty_bar(s), 1);         // tcgen05.commit (multicast to both CTAs)
    }
    for (int a = 0; a < 2; ++a) {
      tc::mbar_init(tfull_bar(a), 1);
      tc::mbar_init(tempty_bar(a), 2 * kEpiWarps);   // epilogue warps of BOTH CTAs (leader's barrier)
    }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc_pair<C::TMEM_COLS>(tc::smem_u32(tmem_ptr));
  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();                          // the peer's barriers exist before any remote signal
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // =================================================== TMA producer
    if (lane == 0) {
      for (int v = 0; v < 4; ++v) tc::tma_prefetch_desc(&maps.a[v]);
      tc::tma_prefetch_desc(&maps.w);
      tc::tma_prefetch_desc(&maps.o);
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile0; tile < total_tiles; tile += tstep) {
        const int nt = nt_of(tile);
        int it = 2 * mp_of(tile) + crank;               // this CTA's M tile (may lie past the end: all zero)
        const int w0 = (it % P.tiles_w) * P.tw; it /= P.tiles_w;
        const int h0 = (it % P.tiles_h) * P.th;
        const int n0 = (it / P.tiles_h) * P.tn;
        int t = 0, cb = 0;
        for (int kb = 0; kb < KB; ++kb) {
          tc::mbar_wait(empty_bar(stage), phase ^ 1);
          C16_TR(0, tr_i); ++tr_i;                       // slot free: loads of this k-block go out
          if (crank == 0) tc::mbar_arrive_expect_tx(full_bar(stage), 2 * C::STAGE);
          const uint32_t lead_bar = tc::mapa(full_bar(stage), 0);
          const uint32_t a_dst = base + stage * C::STAGE;
          const CUtensorMap* am = &maps.a[P.map[t]];
          const int cx = cb * 64, wx = w0 + P.dwq[t], hx = h0 + P.dhq[t];
          tc::tma_load_5d_pair(a_dst, am, lead_bar, cx, wx, hx, n0, 0);
          if (NP == 2) tc::tma_load_5d_pair(a_dst + C::A_PLANE, am, lead_bar, cx, wx, hx, n0, 1);
          const uint32_t b_dst = a_dst + C::A_BYTES;
          const int kx = P.koff[t] + cx, rx = nt * BN + crank * C::BROWS;
          tc::tma_load_3d_pair(b_dst, &maps.w, lead_bar, kx, rx, 0);
          if (NP == 2) tc::tma_load_3d_pair(b_dst + C::B_PLANE, &maps.w, lead_bar, kx, rx, 1);
          if (++cb == P.CB) { cb = 0; ++t; }
          if (++stage == C::S) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // =================================================== MMA issuer (leader CTA)
    if (lane == 0 && crank == 0) {
      constexpr uint32_t idesc = tc::idesc_f16(2 * BM, BN, 0, 0);
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      for (int tile = tile0; tile < total_tiles; tile += tstep) {
        C16_TR(1, tr_i); ++tr_i;                         // (a) ready for the tile
        tc::mbar_wait_cluster(tempty_bar(as), aphase ^ 1);
        tc::tc_fence_after();
        C16_TR(1, tr_i); ++tr_i;                         // (b) accumulator buffer free
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < KB; ++kb) {
          tc::mbar_wait_cluster(full_bar(stage), phase);
          tc::tc_fence_after();
          if (kb == 0) { C16_TR(1, tr_i); ++tr_i; }      // (c) first operands landed
          const uint32_t a_hi = base + stage * C::STAGE;
          const uint32_t b_hi = a_hi + C::A_BYTES;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {               // 4 x K = 16 fp16 (32 bytes)
            const uint64_t ah = tc::desc_kmajor_sw128(a_hi + kk * 32);
            const uint64_t bh = tc::desc_kmajor_sw128(b_hi + kk * 32);
            if (NP == 2) {
              const uint64_t al = tc::desc_kmajor_sw128(a_hi + C::A_PLANE + kk * 32);
              const uint64_t bl = tc::desc_kmajor_sw128(b_hi + C::B_PLANE + kk * 32);
              tc::mma_f16_pair(d_tmem, al, bh, idesc, (kb | kk) != 0);
              tc::mma_f16_pair(d_tmem, ah, bl, idesc, 1);
              tc::mma_f16_pair(d_tmem, ah, bh, idesc, 1);
            } else {
              tc::mma_f16_pair(d_tmem, ah, bh, idesc, (kb | kk) != 0);
            }
          }
          tc::mma_commit_pair(empty_bar(stage));          // frees the slot in both CTAs
          if (++stage == C::S) { stage = 0; phase ^= 1; }
        }
        tc::mma_commit_pair(tfull_bar(as));               // accumulator complete (both CTAs)
        C16_TR(1, tr_i); ++tr_i;                         // (d) all MMAs of the tile issued
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else {
    // =================================================== epilogue (4 warps)
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    const int wq = warp - 2;
    const int et = wq * 32 + lane;             // 0..127
    const bool tr_e = trace_on && wq == 0 && lane == 0;    // the one thread that records the epilogue's events
    uint8_t* stg = epi_stage + wq * 4096;      // this warp's 32 rows x 128 B, SWIZZLE_128B
    const uint32_t stg_u32 = tc::smem_u32(stg);
    float* sst = sstat + wq * 2 * BN;          // this warp's statistics slice, summed over tiles
    const float alpha = in_sc[1] * w_sc[1];
    const int twh = P.tw * P.th;
    // the warp's 32 tile rows are the sub-box (ew, eh, en) of the tile at this offset
    const int r0 = q * 32;
    const int w_off = r0 % P.tw, h_off = (r0 / P.tw) % P.th, n_off = r0 / twh;
    // staged element (row rr, column cc) of the swizzled box
    auto stg_at = [&](int rr, int cc) -> float* {
      return reinterpret_cast<float*>(stg + rr * 128 + ((((cc >> 2) ^ (rr & 7)) << 4) | ((cc & 3) << 2)));
    };
    if (stats) {
      for (int c = lane; c < 2 * BN; c += 32) sst[c] = 0.f;
      __syncwarp();
    }
    auto flush_stats = [&](int nt) {
      // every column below Cout of N tile `nt` carries the sums of all tiles since the last flush
      asm volatile("bar.sync 2, 128;" ::: "memory");
      for (int c = et; c < 2 * BN; c += 128) {
        const int which = c / BN, col = nt * BN + (c % BN);
        if (col < P.Cout) {
          const float v = (sstat[c] + sstat[2 * BN + c]) + (sstat[4 * BN + c] + sstat[6 * BN + c]);
          atomicAdd(stats + (int64_t)which * P.Cout + col, (double)v);
        }
      }
      asm volatile("bar.sync 2, 128;" ::: "memory");
      for (int c = lane; c < 2 * BN; c += 32) sst[c] = 0.f;
      __syncwarp();
    };
    int as = 0, nt_prev = -1;
    uint32_t aphase = 0;
    for (int tile = tile0; tile < total_tiles; tile += tstep) {
      const int nt = nt_of(tile);
      const int mt = 2 * mp_of(tile) + crank;
      if (stats && nt_prev >= 0 && nt != nt_prev) flush_stats(nt_prev);
      nt_prev = nt;
      int it = mt;
      const int w0 = (it % P.tiles_w) * P.tw; it /= P.tiles_w;
      const int h0 = (it % P.tiles_h) * P.th;
      const int n0 = (it / P.tiles_h) * P.tn;
      unsigned vmask = 0;
      if (stats) {
        const int r = r0 + lane;               // tile row == TMEM lane
        const int w = w0 + r % P.tw, h = h0 + (r / P.tw) % P.th, n = n0 + r / twh;
        vmask = __ballot_sync(0xffffffffu, mt < P.m_tiles && w < P.Wp && h < P.Hp && n < P.N);
      }
      if (tr_e) { C16_TR(2, tr_i); ++tr_i; }   // (a) waiting for the accumulator
      tc::mbar_wait(tfull_bar(as), aphase);
      tc::tc_fence_after();
      if (tr_e) { C16_TR(2, tr_i); ++tr_i; }   // (b) accumulator complete
      // chunks of 32 columns.  The TMEM load is issued first and lands while lane 0 waits for the TMA
      // unit to finish reading the previous box.  (Issuing it a chunk ahead was measured and is SLOWER --
      // fence.proxy.async is a MEMBAR.ALL.CTA that waits for a load in flight, and a load in flight behind
      // the statistics' LDS stream costs more than it hides: profiles/r2_conv16_epilogue_probes.md.)
#pragma unroll 1
      for (int chunk = 0; chunk < BN / 32; ++chunk) {
        const int col0 = nt * BN + chunk * 32;
        if (col0 >= P.Cout) break;             // N tail
        uint32_t rg[32];
#ifdef EPB_C16_TRACE_CHUNKS
        if (tr_e) { C16_TR(3, tr_c); ++tr_c; }   // chunk (a) start
#endif
        tc::tmem_ld32(tmem_base + as * BN + chunk * 32 + ((uint32_t)(q * 32) << 16), rg);
        // the previous box must have been read by the TMA unit before it is overwritten
        if (lane == 0) tc::tma_store_wait_read<0>();
#ifdef EPB_C16_TRACE_CHUNKS
        if (tr_e) { C16_TR(3, tr_c); ++tr_c; }   // (b) box free
#endif
        __syncwarp();
        tc::tmem_ld_wait();
#ifdef EPB_C16_TRACE_CHUNKS
        if (tr_e) { C16_TR(3, tr_c); ++tr_c; }   // (c) accumulator columns in registers
#endif
#pragma unroll
        for (int c = 0; c < 32; c += 4) {
          float4 x = make_float4(__uint_as_float(rg[c]) * alpha, __uint_as_float(rg[c + 1]) * alpha,
                                 __uint_as_float(rg[c + 2]) * alpha, __uint_as_float(rg[c + 3]) * alpha);
          if (bias && col0 + c < P.Cout) {
            const float4 b = *reinterpret_cast<const float4*>(bias + col0 + c);
            x.x += b.x; x.y += b.y; x.z += b.z; x.w += b.w;
          }
          *reinterpret_cast<float4*>(stg + lane * 128 + (((c >> 2) ^ (lane & 7)) << 4)) = x;
        }
#ifdef EPB_C16_TRACE_CHUNKS
        if (tr_e) { C16_TR(3, tr_c); ++tr_c; }   // (d) staged
#endif
        tc::fence_proxy_async();               // generic-proxy writes -> visible to the TMA unit
        __syncwarp();
#ifdef EPB_C16_TRACE_CHUNKS
        if (tr_e) { C16_TR(3, tr_c); ++tr_c; }   // (e) fenced
#endif
        if (lane == 0 && mt < P.m_tiles && !(P.probe & 4)) {
          if (P.accumulate)
            tc::tma_reduce_add_4d(&maps.o, stg_u32, col0, w0 + w_off, h0 + h_off, n0 + n_off);
          else
            tc::tma_store_4d(&maps.o, stg_u32, col0, w0 + w_off, h0 + h_off, n0 + n_off);
          tc::tma_store_commit();
        }
#ifdef EPB_C16_TRACE_CHUNKS
        if (tr_e) { C16_TR(3, tr_c); ++tr_c; }   // (f) store issued
#endif
        if (stats && !(P.probe & 8)) {
          // lane = column: sum over the staged valid rows (conflict free: the swizzle spreads
          // the 32 columns of a row over the 32 banks); four partial sums keep the chains short
          float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int rr = 0; rr < 32; ++rr) {
            const float x = ((vmask >> rr) & 1u) ? *stg_at(rr, lane) : 0.f;
            s1[rr & 3] += x;
            s2[rr & 3] = fmaf(x, x, s2[rr & 3]);
          }
          sst[chunk * 32 + lane] += (s1[0] + s1[1]) + (s1[2] + s1[3]);
          sst[BN + chunk * 32 + lane] += (s2[0] + s2[1]) + (s2[2] + s2[3]);
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (tr_e) { C16_TR(2, tr_i); ++tr_i; }   // (c) tile written out
      if (lane == 0) tc::mbar_arrive_cluster_relaxed(tc::mapa(tempty_bar(as), 0));
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (stats && nt_prev >= 0) flush_stats(nt_prev);
    if (lane == 0) tc::tma_store_wait<0>();    // the boxes are written before the CTA exits
    __syncwarp();
  }

  tc::tc_fence_before();
  __syncthreads();
  tc::cluster_sync();             // the peer may still read this CTA's smem / signal its barriers
  if (warp == 1) {
    tc::tc_fence_after();
    tc::tmem_dealloc_pair<C::TMEM_COLS>(tmem_base);
  }
}

template <int BN, int NP>
int launch16(const Plan16& P, const Maps16& maps, const float* in_sc, const float* w_sc,
             const float* bias, float* out, double* stats, cudaStream_t st) {
  using C = Cfg16<BN, NP>;
  static bool attr_set = false;
  if (!attr_set) {
    EPB_CUDA(cudaFuncSetAttribute(conv16_kernel<BN, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  C::SMEM));
    attr_set = true;
  }
  const int64_t pairs = (int64_t)((P.m_tiles + 1) / 2) * P.n_tiles;
  const int grid = 2 * (int)(pairs < kNumSMs / 2 ? pairs : kNumSMs / 2);
  conv16_kernel<BN, NP><<<grid, kThreads16, C::SMEM, st>>>(P, maps, in_sc, w_sc, bias, out, stats);
  EPB_LAUNCH_CHECK();
  return EPB_OK;
}

}  // namespace

// profiling aid: the clock64() trace cluster 0 of the last EPB_C16_PROBE & 32 launch left (4 roles x 2 CTAs x 256)
extern "C" __attribute__((visibility("default"))) int epb_debug_conv16_trace(long long* host_dst, int n) {
  EPB_CHECK_ARG(host_dst && n > 0 && n <= 4 * 2 * 256);
  EPB_CUDA(cudaDeviceSynchronize());
  EPB_CUDA(cudaMemcpyFromSymbol(host_dst, g_c16_trace, (size_t)n * sizeof(long long)));
  return EPB_OK;
}

extern "C" __attribute__((visibility("default"))) int epb_conv16_fprop(
    const epb_conv_geom* g, const epb_half* in, const float* in_sc, const epb_half* w,
    const float* w_sc, const float* bias, float* out, double* stats, int planes,
    epb_stream_t stream) {
  int rc = epb_conv_geom_check(g);
  if (rc) return rc;
  EPB_CHECK_ARG(in && in_sc && w && w_sc && out);
  EPB_CHECK_ARG(planes == 1 || planes == 2);
  EPB_CHECK_ARG(g->Cin % 64 == 0 && g->Cout % 4 == 0 && g->Cout >= 4);
  EPB_CHECK_ARG(g->is == 1 || g->is == 2);
  EPB_CHECK_ARG(!(stats && g->accumulate));
  EPB_CHECK_ARG((reinterpret_cast<uintptr_t>(in) & 127) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0);
  Plan16 P;
  Maps16 maps;
  memset(&maps, 0, sizeof(maps));
  P.Ho = g->Ho; P.Wo = g->Wo; P.Cout = g->Cout; P.os = g->os; P.ph = g->ph; P.pw = g->pw;
  P.T = g->T; P.CB = g->Cin / 64; P.accumulate = g->accumulate;
  // a 1x1 stride-1 layer whose phase grid IS the input and the output grid is a plain
  // [M][C] matrix: tile it as rows (no waste whatever H and W are)
  const bool dense = g->T == 1 && g->is == 1 && g->os == 1 && g->dh[0] == 0 && g->dw[0] == 0 &&
                     g->Hp == g->Hi && g->Wp == g->Wi && g->Hp == g->Ho && g->Wp == g->Wo;
  int N = g->N, Hi = g->Hi, Wi = g->Wi;
  P.N = g->N; P.Hp = g->Hp; P.Wp = g->Wp;
  if (dense) {
    const int64_t M = (int64_t)g->N * g->Hp * g->Wp;
    EPB_CHECK_ARG(M < (1LL << 31));
    N = 1; Hi = 1; Wi = (int)M;
    P.N = 1; P.Hp = 1; P.Wp = (int)M; P.Ho = 1; P.Wo = (int)M;
  }
  epb_choose_tile(P.N, P.Hp, P.Wp, BM, P.tw, P.th, P.tn);
  P.tiles_w = (P.Wp + P.tw - 1) / P.tw;
  P.tiles_h = (P.Hp + P.th - 1) / P.th;
  const int64_t mt = (int64_t)P.tiles_w * P.tiles_h * ((P.N + P.tn - 1) / P.tn);
  EPB_CHECK_ARG(mt < (1LL << 30));
  P.m_tiles = (int)mt;
  bool need[4] = {false, false, false, false};
  for (int t = 0; t < g->T; ++t) {
    int qh, qw, dq_h, dq_w;
    epb_tap_split(g->dh[t], g->is, qh, dq_h);
    epb_tap_split(g->dw[t], g->is, qw, dq_w);
    P.map[t] = (unsigned char)(qh * 2 + qw);
    P.dhq[t] = (short)dq_h;
    P.dwq[t] = (short)dq_w;
    P.koff[t] = g->wt[t] * g->Cin;
    need[qh * 2 + qw] = true;
  }
  for (int v = 0; v < 4; ++v) {
    if (!need[v]) continue;
    rc = epb_make_act_map(&maps.a[v], in, N, Hi, Wi, g->Cin, g->is, v >> 1, v & 1, P.tw, P.th, P.tn,
                          planes);
    if (rc) return rc;
  }
  for (int v = 0; v < 4; ++v)
    if (!need[v]) {                         // unused slots hold a valid map (they are prefetched)
      for (int u = 0; u < 4; ++u)
        if (need[u]) { maps.a[v] = maps.a[u]; break; }
    }
  // tile order: statistics want runs of tiles with the same N tile (one flush per run); without
  // statistics, N-fastest lets the concurrently running tiles of one M tile share its A rows in L2
  P.m_fastest = stats != nullptr;
  // profiling switches (tools/one_conv16.py): 1 flips the tile order, 2 forces the 128-column N tile,
  // 4 / 8 drop the epilogue's stores / statistics (wrong results; never set in a product run)
  static const int probe = getenv("EPB_C16_PROBE") ? atoi(getenv("EPB_C16_PROBE")) : 0;
  P.probe = probe;
  if (probe & 1) P.m_fastest = !P.m_fastest;
  {
    // output box of one epilogue warp: its 32 tile rows as the sub-box (ew, eh, en)
    const int ew = P.tw < 32 ? P.tw : 32;
    const int eh = P.th < 32 / ew ? P.th : 32 / ew;
    const int en = 32 / (ew * eh);
    epb_encode_tiled_fn enc = epb_get_encode_tiled();
    if (!enc) {
      epb_set_error("cuTensorMapEncodeTiled entry point unavailable");
      return EPB_ECUDA;
    }
    const int os = g->os;
    const int Wv = dense ? P.Wp : (g->Wo - g->pw + os - 1) / os, Hv = dense ? 1 : (g->Ho - g->ph + os - 1) / os;
    const int64_t Wo = dense ? P.Wp : g->Wo, Ho = dense ? 1 : g->Ho;
    const cuuint64_t dims[4] = {(cuuint64_t)g->Cout, (cuuint64_t)Wv, (cuuint64_t)Hv, (cuuint64_t)N};
    const cuuint64_t strides[3] = {(cuuint64_t)os * g->Cout * 4, (cuuint64_t)os * Wo * g->Cout * 4,
                                   (cuuint64_t)Ho * Wo * g->Cout * 4};
    const cuuint32_t box[4] = {32, (cuuint32_t)ew, (cuuint32_t)eh, (cuuint32_t)en};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    float* ob = out + ((int64_t)(dense ? 0 : g->ph) * Wo + (dense ? 0 : g->pw)) * g->Cout;
    CUresult cr = enc(&maps.o, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, ob, dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                      CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
      epb_set_error("cuTensorMapEncodeTiled(output %dx%dx%dx%d os %d) failed (%d)", g->N, g->Ho, g->Wo,
                    g->Cout, os, (int)cr);
      return EPB_ECUDA;
    }
  }
  // N tile: 256 unless that wastes more than a quarter of the columns
  int bn;
  if (g->Cout <= 64) bn = 64;
  else if (g->Cout <= 128) bn = 128;
  else {
    const int p256 = (g->Cout + 255) / 256 * 256, p128 = (g->Cout + 127) / 128 * 128;
    bn = (p256 * 4 > p128 * 5) ? 128 : 256;
    if (probe & 2) bn = 128;
  }
  P.n_tiles = (g->Cout + bn - 1) / bn;
  {
    epb_encode_tiled_fn enc = epb_get_encode_tiled();
    if (!enc) {
      epb_set_error("cuTensorMapEncodeTiled entry point unavailable");
      return EPB_ECUDA;
    }
    const int64_t K = (int64_t)g->Tw * g->Cin;
    const cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)g->Cout, (cuuint64_t)planes};
    const cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)K * 2 * g->Cout};
    const cuuint32_t box[3] = {64, (cuuint32_t)(bn / 2), 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult cr = enc(&maps.w, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<epb_half*>(w), dims,
                      strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) {
      epb_set_error("cuTensorMapEncodeTiled(weights %d x %lld) failed (%d)", g->Cout, (long long)K,
                    (int)cr);
      return EPB_ECUDA;
    }
  }
  cudaStream_t st = as_stream(stream);
  if (planes == 1) {
    if (bn == 64) return launch16<64, 1>(P, maps, in_sc, w_sc, bias, out, stats, st);
    if (bn == 128) return launch16<128, 1>(P, maps, in_sc, w_sc, bias, out, stats, st);
    return launch16<256, 1>(P, maps, in_sc, w_sc, bias, out, stats, st);
  }
  if (bn == 64) return launch16<64, 2>(P, maps, in_sc, w_sc, bias, out, stats, st);
  if (bn == 128) return launch16<128, 2>(P, maps, in_sc, w_sc, bias, out, stats, st);
  return launch16<256, 2>(P, maps, in_sc, w_sc, bias, out, stats, st);
}
