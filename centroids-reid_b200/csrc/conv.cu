// Trunk (ResNet50 / ResNet50-IBN-A) inference forward: fused conv + folded-BN (+ residual)
// (+ ReLU) as implicit GEMM on tcgen05 tensor cores, fed by TMA.
//
// Replaces modelling/backbones/resnet.py:51-133, resnet_ibn_a.py:18-141,
// modelling/baseline.py:91-96 and the eval embedding path modelling/bases.py:169-177 /
// inference/inference_utils.py:104-113.
//
// Layout.  Activations NHWC fp16; weights [Cout][kh][kw][Cin] fp16 with the eval-mode
// BatchNorm scale folded in, bias fp32.  GEMM view: D[M = N*Ho*Wo, Cout] = A[M, K] W^T with
// K = kh*kw*Cin.  There is no im2col buffer: an M-tile is a TH x TW block of output pixels
// of one image (TH*TW = 128) and, for every filter tap (r, s) and 64-channel slab, ONE 4-D TMA
// box {64 ch, TW, TH, 1} at (c0, w0 + s - pad, h0 + r - pad, n) lands in shared memory as a
// 128-row x 128-byte K-major operand tile (SWIZZLE_128B); out-of-bounds coordinates are
// zero-filled by the TMA unit, which IS the convolution's zero padding.  Stride-2 convolutions
// read four parity views {h%2, w%2} of the input (strided tensor maps), so every box is still a
// dense stride-1 box.  Accumulators live in TMEM (double-buffered), the epilogue applies
// bias / residual / ReLU and writes fp16 NHWC.
//
// Roofline: tensor pipe for the 3x3 and wide 1x1 convolutions, HBM for the narrow 1x1s
// (arithmetic intensity 2*Cin*Cout/(2*(Cin+Cout)) flop/B < 221); algorithmic bytes per conv =
// 2*(M*Cin [if read once] + M*Cout [+ M*Cout residual]) + 2*K*Cout.
#include <stdlib.h>

#include <algorithm>

#include "common.h"
#include "umma.cuh"

namespace ctl {

static constexpr int CBM = 128;  // output pixels per tile
static constexpr int CBK = 64;   // channels per k-block (128 bytes)
static constexpr int CONV_THREADS = 320;  // TMA warp, MMA warp, 8 epilogue warps
static constexpr int A_TILE_BYTES = CBM * CBK * 2;

struct ConvTap {
  int map;      // which A tensor map (parity view, or the second source of a K-concatenated 1x1)
  int dh, dw;
  int koff;     // offset of this tap's channel slab inside the weight K dimension
  int cblocks;  // 64-channel slabs of this tap (its source's Cin / 64)
};

struct ConvKernelParams {
  CUtensorMap a_map[4];
  CUtensorMap b_map;
  CUtensorMap out_map;  // NHWC output, box {64 ch, TW, TH, 1}
  CUtensorMap res_map;  // residual, same geometry
  ConvTap taps[9];
  int n_taps;
  int k_blocks;  // sum of the taps' cblocks = K / 64
  int n_img, Ho, Wo, Cout;
  int TW, TH, tiles_w, tiles_h;
  int m_tiles, n_tiles;
  const float* bias;        // [Cout]
  int has_residual;
  int relu;                 // apply ReLU to channels >= relu_from
  int relu_from;
};

template <int BN>
struct ConvCfg {
  static constexpr int B_TILE_BYTES = BN * CBK * 2;
  static constexpr int STAGE_BYTES = A_TILE_BYTES + B_TILE_BYTES;
  static constexpr int STAGES = BN == 64 ? 5 : (BN == 128 ? 4 : 3);
  static constexpr int TMEM_COLS = BN == 64 ? 128 : (BN == 128 ? 256 : 512);  // 2 accumulator stages
  static constexpr int OUT_SLABS = 4;                  // [128 px][64 ch] fp16 staging slabs for the TMA stores
  static constexpr int IDENT_BYTES = 64 * CBK * 2;     // 64x64 identity operand (residual add on the tensor core)
  static constexpr int BIAS_BYTES = 2048 * 4;          // the layer's whole bias vector (Cout <= 2048), loaded once
  static constexpr size_t SMEM =
      (size_t)STAGES * STAGE_BYTES + OUT_SLABS * A_TILE_BYTES + IDENT_BYTES + BIAS_BYTES + 1024 + 256;
};

// Tile order: n fastest, then pixel tiles row-major inside an image, then images.  Each CTA owns a
// CONTIGUOUS range of tiles so that coordinates advance by carries (no integer division in the loop)
// and consecutive tiles of a CTA reuse the same activation tile from L2.
struct TileIter {
  int nt, tw, th, img;
  __device__ __forceinline__ void init(int tile, const ConvKernelParams& p) {
    const int mt = tile / p.n_tiles;
    nt = tile - mt * p.n_tiles;
    const int per_img = p.tiles_w * p.tiles_h;
    img = mt / per_img;
    const int tr = mt - img * per_img;
    th = tr / p.tiles_w;
    tw = tr - th * p.tiles_w;
  }
  __device__ __forceinline__ void next(const ConvKernelParams& p) {
    if (++nt == p.n_tiles) {
      nt = 0;
      if (++tw == p.tiles_w) {
        tw = 0;
        if (++th == p.tiles_h) {
          th = 0;
          ++img;
        }
      }
    }
  }
};

template <int BN>
__global__ void __launch_bounds__(CONV_THREADS, 1) conv_gemm_kernel(const __grid_constant__ ConvKernelParams p) {
  using Cfg = ConvCfg<BN>;
  constexpr int NSUB = BN / 64;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t out_stage = smem_base + Cfg::STAGES * Cfg::STAGE_BYTES;
  const uint32_t ident = out_stage + Cfg::OUT_SLABS * A_TILE_BYTES;
  const uint32_t bias_sm = ident + Cfg::IDENT_BYTES;
  const uint32_t bar_base = bias_sm + Cfg::BIAS_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::STAGES + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * Cfg::STAGES + 4);
  uint8_t* gsm = smem_raw + (smem_base - smem_u32(smem_raw));  // generic view of the aligned arena

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = p.m_tiles * p.n_tiles;
  const int conv_kblocks = p.k_blocks;
  // contiguous, balanced tile range of this CTA
  const int per = num_tiles / (int)gridDim.x, rem = num_tiles - per * (int)gridDim.x;
  const int t_begin = (int)blockIdx.x * per + min((int)blockIdx.x, rem);
  const int t_end = t_begin + per + ((int)blockIdx.x < rem ? 1 : 0);

  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 8);
    }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.a_map[i]);
    tma_prefetch_desc(&p.b_map);
    tma_prefetch_desc(&p.out_map);
    tma_prefetch_desc(&p.res_map);
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  for (int i = threadIdx.x; i < p.Cout; i += blockDim.x)
    reinterpret_cast<float*>(gsm + (bias_sm - smem_base))[i] = p.bias[i];
  {  // 64x64 fp16 identity, K-major, SWIZZLE_128B: row r holds a single 1.0 at k = r
    uint8_t* id = gsm + (ident - smem_base);
    for (int i = threadIdx.x; i < Cfg::IDENT_BYTES / 16; i += blockDim.x) reinterpret_cast<uint4*>(id)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    if (threadIdx.x < 64) {
      const int r = threadIdx.x;
      *reinterpret_cast<__half*>(id + r * 128 + (((r >> 3) ^ (r & 7)) << 4) + (r & 7) * 2) = __float2half(1.f);
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();  // the next kernel may begin its prologue
  pdl_wait();               // activations of the previous kernel are complete and visible
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0 && t_begin < t_end) {
      int stage = 0;
      uint32_t phase = 0;
      TileIter it;
      it.init(t_begin, p);
      for (int tile = t_begin; tile < t_end; ++tile, it.next(p)) {
        const int h0 = it.th * p.TH, w0 = it.tw * p.TW;
        for (int t = 0; t < p.n_taps; ++t) {
          const ConvTap tap = p.taps[t];
          for (int cb = 0; cb < tap.cblocks; ++cb) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            const uint32_t dst = smem_base + stage * Cfg::STAGE_BYTES;
            mbar_arrive_expect_tx(full_bar(stage), Cfg::STAGE_BYTES);
            tma_load_4d(dst, &p.a_map[tap.map], full_bar(stage), cb * CBK, w0 + tap.dw, h0 + tap.dh, it.img);
            tma_load_2d(dst + A_TILE_BYTES, &p.b_map, full_bar(stage), tap.koff + cb * CBK, it.nt * BN);
            if (++stage == Cfg::STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
        if (p.has_residual) {
          // the residual rides the same ring: one [128 px][64 ch] slab per 64 output channels,
          // added to the accumulator by an identity MMA (exact: fp16 x 1.0 into fp32)
          for (int j = 0; j < NSUB; ++j) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            mbar_arrive_expect_tx(full_bar(stage), A_TILE_BYTES);
            tma_load_4d(smem_base + stage * Cfg::STAGE_BYTES, &p.res_map, full_bar(stage), it.nt * BN + j * 64, w0, h0,
                        it.img);
            if (++stage == Cfg::STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(CBM, BN);
      constexpr uint32_t idesc64 = make_idesc_f16(CBM, 64);
      const uint64_t d_ident = make_sw128_kmajor_desc(ident);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = t_begin; tile < t_end; ++tile) {
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        tc_fence_after();
        const uint32_t acc = tmem_base + as * BN;
        for (int kb = 0; kb < conv_kblocks; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t base = smem_base + stage * Cfg::STAGE_BYTES;
          const uint64_t da = make_sw128_kmajor_desc(base);
          const uint64_t db = make_sw128_kmajor_desc(base + A_TILE_BYTES);
#pragma unroll
          for (int k = 0; k < CBK / 16; ++k)
            umma_f16(acc, desc_advance_k(da, k), desc_advance_k(db, k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(empty_bar(stage));
          if (++stage == Cfg::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if (p.has_residual) {
          for (int j = 0; j < NSUB; ++j) {
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            const uint64_t da = make_sw128_kmajor_desc(smem_base + stage * Cfg::STAGE_BYTES);
#pragma unroll
            for (int k = 0; k < CBK / 16; ++k)
              umma_f16(acc + j * 64, desc_advance_k(da, k), desc_advance_k(d_ident, k), idesc64, 1u);
            umma_commit(empty_bar(stage));
            if (++stage == Cfg::STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
        umma_commit(tfull_bar(as));
        if (++as == 2) {
          as = 0;
          aphase ^= 1u;
        }
      }
    }
  } else {
    // ===== epilogue: 8 warps (two per 32-lane TMEM quarter, splitting the columns).  The
    // accumulator (conv + residual) is drained in 64-channel sub-tiles: TMEM -> registers ->
    // (+bias, ReLU) -> fp16 -> swizzled staging slab -> one TMA store per sub-tile; four slabs
    // keep up to three stores in flight.  No global memory access is issued by these warps
    // except the per-tile bias slice.
    const int ew = warp - 2;              // 0..7
    const int et = threadIdx.x - 64;      // 0..255
    const int quarter = warp & 3;         // TMEM lane quarter this warp may read
    const int chalf = ew >> 2;            // which 32-channel half of every 64-channel sub-tile
    const int pix = quarter * 32 + lane;  // pixel inside the tile == TMEM lane == staging row
    const bool leader = (ew == 0 && lane == 0);
    const uint32_t row_off = pix * 128;
    const uint32_t sw = pix & 7;
    uint8_t* oslabs = gsm + (out_stage - smem_base);
    float* bias_s = reinterpret_cast<float*>(gsm + (bias_sm - smem_base));
    int as = 0;
    uint32_t aphase = 0;
    uint32_t g = 0;  // running sub-tile counter -> staging slab
    TileIter it;
    if (t_begin < t_end) it.init(t_begin, p);
    for (int tile = t_begin; tile < t_end; ++tile, it.next(p)) {
      const int h0 = it.th * p.TH, w0 = it.tw * p.TW;
      const float* bias_t = bias_s + it.nt * BN;  // whole bias vector staged in the prologue
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      const uint32_t t0 = tmem_base + as * BN + (static_cast<uint32_t>(quarter * 32) << 16) + chalf * 32;
#pragma unroll 1
      for (int j = 0; j < NSUB; ++j, ++g) {
        const uint32_t b = g & (Cfg::OUT_SLABS - 1);
        const int ch0 = j * 64 + chalf * 32;  // first of this thread's 32 channels inside the n-tile
        uint32_t r[32];
        tmem_ld16(t0 + j * 64, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
        tmem_ld16(t0 + j * 64 + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
        // slab b was handed to a TMA store OUT_SLABS sub-tiles ago: wait until that store has read it
        if (leader) tma_store_wait_read<Cfg::OUT_SLABS - 1>();
        named_bar_sync(1, 256);  // also publishes this tile's bias slice
        tmem_ld_wait();
        if (j == NSUB - 1) {  // last TMEM read of this accumulator stage: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tempty_bar(as));
        }
        uint8_t* oslab = oslabs + b * A_TILE_BYTES + row_off;
        const bool do_relu = p.relu && (it.nt * BN + ch0) >= p.relu_from;  // relu_from is a multiple of 32
#pragma unroll
        for (int c = 0; c < 4; ++c) {  // four 16-byte chunks = 32 channels
          const float4 b0 = *reinterpret_cast<const float4*>(bias_t + ch0 + c * 8);
          const float4 b1 = *reinterpret_cast<const float4*>(bias_t + ch0 + c * 8 + 4);
          float v[8];
          v[0] = __uint_as_float(r[c * 8 + 0]) + b0.x;
          v[1] = __uint_as_float(r[c * 8 + 1]) + b0.y;
          v[2] = __uint_as_float(r[c * 8 + 2]) + b0.z;
          v[3] = __uint_as_float(r[c * 8 + 3]) + b0.w;
          v[4] = __uint_as_float(r[c * 8 + 4]) + b1.x;
          v[5] = __uint_as_float(r[c * 8 + 5]) + b1.y;
          v[6] = __uint_as_float(r[c * 8 + 6]) + b1.z;
          v[7] = __uint_as_float(r[c * 8 + 7]) + b1.w;
          if (do_relu) {
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = fmaxf(v[q], 0.f);
          }
          uint4 o;
          __half2* po = reinterpret_cast<__half2*>(&o);
#pragma unroll
          for (int q = 0; q < 4; ++q) po[q] = __floats2half2_rn(v[2 * q], v[2 * q + 1]);
          *reinterpret_cast<uint4*>(oslab + (((uint32_t)(chalf * 4 + c) ^ sw) << 4)) = o;
        }
        fence_proxy_async();     // staging writes (generic proxy) -> visible to the TMA store (async proxy)
        named_bar_sync(1, 256);  // slab complete
        if (leader) {
          tma_store_4d(&p.out_map, out_stage + b * A_TILE_BYTES, it.nt * BN + j * 64, w0, h0, it.img);
          tma_store_commit();
        }
      }
      if (++as == 2) {
        as = 0;
        aphase ^= 1u;
      }
    }
    if (leader) tma_store_wait<0>();  // shared memory must outlive the last stores
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2) for the compute-bound wide convolutions.
//
// Two CTAs of a cluster own two neighbouring 128-pixel tiles and the SAME 256 output channels.
// CTA 0 issues one tcgen05.mma.cta_group::2 (M = 256, N = 256) per 16-wide k-step: rows 0-127 of A
// come from CTA 0's shared memory, rows 128-255 from CTA 1's; each CTA stages only HALF of the weight
// tile (128 of the 256 output channels).  Per CTA and k-block that is 16 KiB of activations + 16 KiB of
// weights instead of 16 + 32 KiB: the shared-memory fill rate (~50-60 B/clk/SM measured), not the
// tensor pipe, is what bounds the single-CTA kernel on these layers.
// Protocol: both producers credit their TMA bytes to CTA 0's `full` barrier; the leader's commits are
// multicast to both CTAs' `empty` / `tmem_full` barriers; both epilogues release the accumulator
// stage on CTA 0's `tmem_empty` barrier.  Each CTA drains its own 128 TMEM lanes.
// ---------------------------------------------------------------------------------------
// VAR selects the shared-memory split (the total is the 227 KiB of one SM):
//   1: non-residual layers -- 5 operand stages (6 for 128-wide tiles) + 2 output staging slabs
//      (measured 2.5-3 % faster than 4 + 4 on the bs-256 trunk);
//   2: residual layers     -- 4 (5) operand stages + 5 staging slabs that double as residual landing
//      buffers: the residual tile is TMA-loaded INTO the staging slab three sub-tiles ahead, the
//      epilogue adds it in place (ld.shared / add / st.shared on the thread's own 64 bytes) and the
//      same slab is TMA-stored.  Round 1 added the residual with an identity MMA through the operand
//      ring, which cost 16 N=64 MMAs per 256x256 tile (25 % of the tensor time of a K=512 layer).
template <int BN_, int VAR_ = 1>
struct PairCfg {
  static constexpr int BN = BN_;                                  // 256 or 128 output channels per pair tile
  static constexpr bool RES = VAR_ == 2;
  static constexpr int B_HALF_BYTES = (BN / 2) * CBK * 2;         // this CTA's half of the weight tile: 16 / 8 KiB
  static constexpr int STAGE_BYTES = A_TILE_BYTES + B_HALF_BYTES;  // 32 / 24 KiB
  static constexpr int STAGES = (BN == 256 ? 4 : 5) + (RES ? 0 : 1);
  static constexpr int TMEM_COLS = 2 * BN;                        // two accumulator stages
  static constexpr int OUT_SLABS = RES ? 5 : 2;
  static constexpr int RES_AHEAD = 3;                             // residual prefetch distance, sub-tiles
  static constexpr int BIAS_BYTES = 2048 * 4;  // the layer's whole bias vector, loaded once
  static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + OUT_SLABS * A_TILE_BYTES + BIAS_BYTES + 1024 + 256;
};

// pair tile -> (n tile, this CTA's 128-pixel tile); n fastest.  Coordinates advance by carries: one set of
// integer divisions per role, not per tile.
struct PairIter {
  int nt, w_t, h_t, img;
  __device__ __forceinline__ void init(int tile, const ConvKernelParams& q, int rank_, int per_img) {
    const int pm = tile / q.n_tiles;
    nt = tile - pm * q.n_tiles;
    const int mt = 2 * pm + rank_;
    img = mt / per_img;
    const int tr = mt - img * per_img;
    h_t = tr / q.tiles_w;
    w_t = tr - h_t * q.tiles_w;
  }
  __device__ __forceinline__ void next(const ConvKernelParams& q) {
    if (++nt < q.n_tiles) return;
    nt = 0;
    w_t += 2;  // the pair advances by two 128-pixel tiles
    while (w_t >= q.tiles_w) {
      w_t -= q.tiles_w;
      if (++h_t == q.tiles_h) {
        h_t = 0;
        ++img;
      }
    }
  }
};

template <int BN_T, int VAR_T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CONV_THREADS, 1)
    conv_gemm_pair_kernel(const __grid_constant__ ConvKernelParams p) {
  using Cfg = PairCfg<BN_T, VAR_T>;
  constexpr int BN = Cfg::BN;
  constexpr int NSUB = BN / 64;
  constexpr int SLABS = Cfg::OUT_SLABS;
  constexpr int RES_WAIT = Cfg::RES ? SLABS - Cfg::RES_AHEAD - 1 : 0;  // stores that may still be reading their slab
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t out_stage = smem_base + Cfg::STAGES * Cfg::STAGE_BYTES;
  const uint32_t bias_sm = out_stage + SLABS * A_TILE_BYTES;
  const uint32_t bar_base = bias_sm + Cfg::BIAS_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };                         // used in CTA 0 only
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::STAGES + s); };         // per CTA
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::STAGES + s); };     // per CTA
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::STAGES + 2 + s); };  // used in CTA 0 only
  auto res_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::STAGES + 4 + s); };   // per CTA: residual landed in slab s
  const uint32_t tmem_slot = bar_base + 8u * (2 * Cfg::STAGES + 4 + SLABS);
  uint8_t* gsm = smem_raw + (smem_base - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool is_leader = rank == 0;
  const int n_clusters = (int)gridDim.x >> 1, cid = (int)blockIdx.x >> 1;
  const int m_pairs = p.m_tiles >> 1;
  const int num_tiles = m_pairs * p.n_tiles;  // pair tiles
  const int conv_kblocks = p.k_blocks;
  const int per = num_tiles / n_clusters, rem = num_tiles - per * n_clusters;
  const int t_begin = cid * per + min(cid, rem);
  const int t_end = t_begin + per + (cid < rem ? 1 : 0);
  const int tiles_per_img = p.tiles_w * p.tiles_h;

  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::STAGES; ++s) {
      mbar_init(full_bar(s), 2);   // one arrive per producer of the pair (+ both CTAs' TMA bytes)
      mbar_init(empty_bar(s), 1);  // leader's multicast commit
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);    // leader's multicast commit
      mbar_init(tempty_bar(s), 16);  // 8 epilogue warps of each CTA
    }
    for (int s = 0; s < SLABS; ++s) mbar_init(res_bar(s), 1);
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 4; ++i) tma_prefetch_desc(&p.a_map[i]);
    tma_prefetch_desc(&p.b_map);
    tma_prefetch_desc(&p.out_map);
    tma_prefetch_desc(&p.res_map);
  }
  if (warp == 1) tmem_alloc2<Cfg::TMEM_COLS>(tmem_slot);
  for (int i = threadIdx.x; i < p.Cout; i += blockDim.x)
    reinterpret_cast<float*>(gsm + (bias_sm - smem_base))[i] = p.bias[i];
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // barriers of both CTAs initialised before any remote arrive / TMA credit
  tc_fence_after();
  pdl_launch_dependents();  // the next kernel may begin its prologue
  pdl_wait();               // activations of the previous kernel are complete and visible
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      PairIter it;
      if (t_begin < t_end) it.init(t_begin, p, (int)rank, tiles_per_img);
      for (int tile = t_begin; tile < t_end; ++tile, it.next(p)) {
        const int nt = it.nt, w0 = it.w_t * p.TW, h0 = it.h_t * p.TH, img = it.img;
        for (int t = 0; t < p.n_taps; ++t) {
          const ConvTap tap = p.taps[t];
          for (int cb = 0; cb < tap.cblocks; ++cb) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            const uint32_t dst = smem_base + stage * Cfg::STAGE_BYTES;
            if (is_leader) mbar_arrive_expect_tx(full_bar(stage), 2 * Cfg::STAGE_BYTES);
            else mbar_arrive_cta0(full_bar(stage));
            tma2_load_4d(dst, &p.a_map[tap.map], full_bar(stage), cb * CBK, w0 + tap.dw, h0 + tap.dh, img);
            tma2_load_2d(dst + A_TILE_BYTES, &p.b_map, full_bar(stage), tap.koff + cb * CBK,
                         nt * BN + (int)rank * (BN / 2));
            if (++stage == Cfg::STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (is_leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(256, BN);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = t_begin; tile < t_end; ++tile) {
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        tc_fence_after();
        const uint32_t acc = tmem_base + as * BN;
        for (int kb = 0; kb < conv_kblocks; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t base = smem_base + stage * Cfg::STAGE_BYTES;
          const uint64_t da = make_sw128_kmajor_desc(base);
          const uint64_t db = make_sw128_kmajor_desc(base + A_TILE_BYTES);
#pragma unroll
          for (int k = 0; k < CBK / 16; ++k)
            umma2_f16(acc, desc_advance_k(da, k), desc_advance_k(db, k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma2_commit_mc(empty_bar(stage), 3);
          if (++stage == Cfg::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma2_commit_mc(tfull_bar(as), 3);
        if (++as == 2) {
          as = 0;
          aphase ^= 1u;
        }
      }
    }
  } else {
    // ===================== epilogue (both CTAs, own 128 TMEM lanes) =====================
    // Per 64-channel sub-tile: TMEM -> registers -> (+bias, +residual from the staging slab, ReLU) -> fp16 ->
    // swizzled staging slab -> one TMA store.  No global memory access is issued by these warps.
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int chalf = ew >> 2;
    const int pix = quarter * 32 + lane;
    const bool leader_thread = (ew == 0 && lane == 0);
    const uint32_t row_off = pix * 128;
    const uint32_t sw = pix & 7;
    uint8_t* oslabs = gsm + (out_stage - smem_base);
    float* bias_s = reinterpret_cast<float*>(gsm + (bias_sm - smem_base));
    const bool with_res = Cfg::RES && p.has_residual;
    int as = 0;
    uint32_t aphase = 0;
    int b = 0;            // staging slab of the current sub-tile
    uint32_t bphase = 0;  // parity of res_bar(b)
    // residual prefetch state (leader thread): the sub-tile RES_AHEAD ahead of the one being drained
    PairIter pit;
    int ptile = t_begin, pj = 0, pb = 0;
    auto prefetch_res = [&]() {
      if (ptile < t_end) {
        mbar_arrive_expect_tx(res_bar(pb), A_TILE_BYTES);
        tma_load_4d(out_stage + pb * A_TILE_BYTES, &p.res_map, res_bar(pb), pit.nt * BN + pj * 64, pit.w_t * p.TW,
                    pit.h_t * p.TH, pit.img);
        if (++pb == SLABS) pb = 0;
        if (++pj == NSUB) {
          pj = 0;
          ++ptile;
          pit.next(p);
        }
      }
    };
    if (with_res && leader_thread && t_begin < t_end) {
      pit.init(t_begin, p, (int)rank, tiles_per_img);
      for (int i = 0; i < Cfg::RES_AHEAD; ++i) prefetch_res();
    }
    PairIter it;
    if (t_begin < t_end) it.init(t_begin, p, (int)rank, tiles_per_img);
    for (int tile = t_begin; tile < t_end; ++tile, it.next(p)) {
      const int nt = it.nt, w0 = it.w_t * p.TW, h0 = it.h_t * p.TH, img = it.img;
      const float* bias_t = bias_s + nt * BN;  // whole bias vector staged in the prologue
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      const uint32_t t0 = tmem_base + as * BN + (static_cast<uint32_t>(quarter * 32) << 16) + chalf * 32;
#pragma unroll 1
      for (int j = 0; j < NSUB; ++j) {
        const int ch0 = j * 64 + chalf * 32;
        uint32_t r[32];
        tmem_ld16(t0 + j * 64, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
        tmem_ld16(t0 + j * 64 + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
        if (with_res) {
          // the slab RES_AHEAD sub-tiles ahead was stored SLABS - RES_AHEAD sub-tiles ago: once that store has
          // read it, the next residual tile may land there
          if (leader_thread) {
            tma_store_wait_read<RES_WAIT>();
            prefetch_res();
          }
          mbar_wait(res_bar(b), bphase);  // this sub-tile's residual is in slab b (which is therefore free)
        } else {
          // slab b was handed to a TMA store SLABS sub-tiles ago: wait until that store has read it
          if (leader_thread) tma_store_wait_read<SLABS - 1>();
          named_bar_sync(1, 256);
        }
        tmem_ld_wait();
        if (j == NSUB - 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cta0(tempty_bar(as));
        }
        uint8_t* oslab = oslabs + b * A_TILE_BYTES + row_off;
        const bool do_relu = p.relu && (nt * BN + ch0) >= p.relu_from;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4* slot = reinterpret_cast<uint4*>(oslab + (((uint32_t)(chalf * 4 + c) ^ sw) << 4));
          const float4 b0 = *reinterpret_cast<const float4*>(bias_t + ch0 + c * 8);
          const float4 b1 = *reinterpret_cast<const float4*>(bias_t + ch0 + c * 8 + 4);
          float v[8];
          v[0] = __uint_as_float(r[c * 8 + 0]) + b0.x;
          v[1] = __uint_as_float(r[c * 8 + 1]) + b0.y;
          v[2] = __uint_as_float(r[c * 8 + 2]) + b0.z;
          v[3] = __uint_as_float(r[c * 8 + 3]) + b0.w;
          v[4] = __uint_as_float(r[c * 8 + 4]) + b1.x;
          v[5] = __uint_as_float(r[c * 8 + 5]) + b1.y;
          v[6] = __uint_as_float(r[c * 8 + 6]) + b1.z;
          v[7] = __uint_as_float(r[c * 8 + 7]) + b1.w;
          if (with_res) {
            const uint4 rv = *slot;
            const __half2* rh = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float2 f = __half22float2(rh[q]);
              v[2 * q] += f.x;
              v[2 * q + 1] += f.y;
            }
          }
          if (do_relu) {
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = fmaxf(v[q], 0.f);
          }
          uint4 o;
          __half2* po = reinterpret_cast<__half2*>(&o);
#pragma unroll
          for (int q = 0; q < 4; ++q) po[q] = __floats2half2_rn(v[2 * q], v[2 * q + 1]);
          *slot = o;
        }
        fence_proxy_async();
        named_bar_sync(1, 256);
        if (leader_thread) {
          tma_store_4d(&p.out_map, out_stage + b * A_TILE_BYTES, nt * BN + j * 64, w0, h0, img);
          tma_store_commit();
        }
        if (++b == SLABS) {
          b = 0;
          bphase ^= 1u;
        }
      }
      if (++as == 2) {
        as = 0;
        aphase ^= 1u;
      }
    }
    if (leader_thread) tma_store_wait<0>();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer's shared memory / barriers stay valid until both CTAs are done
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc2<Cfg::TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------
// 3x3 / stride 1 / 64 -> 64 channels (layer1.conv2, the most fill-bound layer of the trunk: the
// generic kernel re-reads the activation tile once per filter tap, 216 KiB of shared-memory fill
// for 9.4 MFLOP).  Here the 9 x [64 x 64] weight slabs (72 KiB) stay RESIDENT in shared memory and
// each 16 x 8 output tile loads ONE halo slab -- 18 rows x 16 pixel lines x 128 B, i.e. the 18 x 10
// halo padded to a 2 KiB row pitch -- by a single TMA box; the nine taps are nine SHIFTED VIEWS of
// that slab: descriptor start = slab + (r*16 + s)*128 B, 8-row groups 2 KiB apart (one output row
// each).  MEASURED on B200: the tensor core derives the 128-byte-swizzle XOR from the absolute
// shared-memory address bits [7,10) -- exactly what the TMA unit used when it wrote the slab -- so
// a start address shifted by whole 128-byte lines needs NO descriptor base_offset (base_offset = s
// gives wrong results; tests/test_trunk_gpu.py::test_conv_shapes[case3] pins this).  36 KiB of fill
// per tile instead of 216 KiB.
// ---------------------------------------------------------------------------------------
static constexpr int C64_HALO_BYTES = 18 * 16 * 128;  // 36 KiB
static constexpr int C64_W_BYTES = 9 * 64 * 128;      // 72 KiB
static constexpr int C64_HALOS = 2;
static constexpr int C64_OUT_SLABS = 4;
static constexpr size_t C64_SMEM = C64_W_BYTES + C64_HALOS * C64_HALO_BYTES + C64_OUT_SLABS * A_TILE_BYTES + 512 + 1024 + 256;

struct C64Params {
  CUtensorMap x_map;    // NHWC input, box {64, 16, 18, 1}
  CUtensorMap w_map;    // [64][576] weights, box {64, 64}
  CUtensorMap out_map;  // NHWC output, box {64, 8, 16, 1}
  const float* bias;
  int n_img, H, W, tiles_h, tiles_w, relu, use_base_offset;
};

__global__ void __launch_bounds__(CONV_THREADS, 1) conv3x3_c64_kernel(const __grid_constant__ C64Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_sm = smem_base;
  const uint32_t halo_sm = w_sm + C64_W_BYTES;
  const uint32_t out_stage = halo_sm + C64_HALOS * C64_HALO_BYTES;
  const uint32_t bias_sm = out_stage + C64_OUT_SLABS * A_TILE_BYTES;
  const uint32_t bar_base = bias_sm + 512;
  const uint32_t w_bar = bar_base;
  auto full_bar = [&](int s) { return bar_base + 8u * (1 + s); };
  auto empty_bar = [&](int s) { return bar_base + 8u * (1 + C64_HALOS + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (1 + 2 * C64_HALOS + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (3 + 2 * C64_HALOS + s); };
  const uint32_t tmem_slot = bar_base + 8u * (5 + 2 * C64_HALOS);
  uint8_t* gsm = smem_raw + (smem_base - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_per_img = p.tiles_h * p.tiles_w;
  const int num_tiles = p.n_img * tiles_per_img;
  const int per = num_tiles / (int)gridDim.x, rem = num_tiles - per * (int)gridDim.x;
  const int t_begin = (int)blockIdx.x * per + min((int)blockIdx.x, rem);
  const int t_end = t_begin + per + ((int)blockIdx.x < rem ? 1 : 0);
  auto coords = [&](int tile, int& w0, int& h0, int& img) {
    img = tile / tiles_per_img;
    const int tr = tile - img * tiles_per_img;
    h0 = (tr / p.tiles_w) * 16;
    w0 = (tr % p.tiles_w) * 8;
  };
  if (threadIdx.x == 0) {
    mbar_init(w_bar, 1);
    for (int s = 0; s < C64_HALOS; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 8);
    }
    fence_barrier_init();
    tma_prefetch_desc(&p.x_map);
    tma_prefetch_desc(&p.w_map);
    tma_prefetch_desc(&p.out_map);
  }
  if (warp == 1) tmem_alloc<128>(tmem_slot);
  if (threadIdx.x >= 64 && threadIdx.x < 128) reinterpret_cast<float*>(gsm + (bias_sm - smem_base))[threadIdx.x - 64] = p.bias[threadIdx.x - 64];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();  // the next kernel may begin its prologue
  pdl_wait();               // activations of the previous kernel are complete and visible
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(w_bar, C64_W_BYTES);
      for (int t = 0; t < 9; ++t) tma_load_2d(w_sm + t * 64 * 128, &p.w_map, w_bar, t * 64, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = t_begin; tile < t_end; ++tile) {
        int w0, h0, img;
        coords(tile, w0, h0, img);
        mbar_wait(empty_bar(stage), phase ^ 1u);
        mbar_arrive_expect_tx(full_bar(stage), C64_HALO_BYTES);
        tma_load_4d(halo_sm + stage * C64_HALO_BYTES, &p.x_map, full_bar(stage), 0, w0 - 1, h0 - 1, img);
        if (++stage == C64_HALOS) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(128, 64);
      mbar_wait(w_bar, 0);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = t_begin; tile < t_end; ++tile) {
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        mbar_wait(full_bar(stage), phase);
        tc_fence_after();
        const uint32_t slab = halo_sm + stage * C64_HALO_BYTES;
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const int r = t / 3, s = t - 3 * r;
          const uint32_t a0 = slab + (r * 16 + s) * 128;
          const uint64_t da = make_sw128_kmajor_desc_ex(a0, 2048, p.use_base_offset ? ((a0 >> 7) & 7u) : 0u);
          const uint64_t db = make_sw128_kmajor_desc(w_sm + t * 64 * 128);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16(tmem_base + as * 64, desc_advance_k(da, k), desc_advance_k(db, k), idesc, (t | k) ? 1u : 0u);
        }
        umma_commit(empty_bar(stage));
        umma_commit(tfull_bar(as));
        if (++stage == C64_HALOS) {
          stage = 0;
          phase ^= 1u;
        }
        if (++as == 2) {
          as = 0;
          aphase ^= 1u;
        }
      }
    }
  } else {
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int chalf = ew >> 2;
    const int pix = quarter * 32 + lane;  // output pixel (row = pix / 8, col = pix % 8) == TMEM lane
    const bool leader = (ew == 0 && lane == 0);
    const uint32_t row_off = pix * 128, sw = pix & 7;
    uint8_t* oslabs = gsm + (out_stage - smem_base);
    const float* bias_s = reinterpret_cast<const float*>(gsm + (bias_sm - smem_base));
    int as = 0;
    uint32_t aphase = 0, g = 0;
    for (int tile = t_begin; tile < t_end; ++tile, ++g) {
      int w0, h0, img;
      coords(tile, w0, h0, img);
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      const uint32_t b = g & (C64_OUT_SLABS - 1);
      uint32_t r[32];
      const uint32_t t0 = tmem_base + as * 64 + (static_cast<uint32_t>(quarter * 32) << 16) + chalf * 32;
      tmem_ld16(t0, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
      tmem_ld16(t0 + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
      if (leader) tma_store_wait_read<C64_OUT_SLABS - 1>();
      named_bar_sync(1, 256);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
      uint8_t* oslab = oslabs + b * A_TILE_BYTES + row_off;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float4 b0 = *reinterpret_cast<const float4*>(bias_s + chalf * 32 + c * 8);
        const float4 b1 = *reinterpret_cast<const float4*>(bias_s + chalf * 32 + c * 8 + 4);
        float v[8] = {__uint_as_float(r[c * 8 + 0]) + b0.x, __uint_as_float(r[c * 8 + 1]) + b0.y,
                      __uint_as_float(r[c * 8 + 2]) + b0.z, __uint_as_float(r[c * 8 + 3]) + b0.w,
                      __uint_as_float(r[c * 8 + 4]) + b1.x, __uint_as_float(r[c * 8 + 5]) + b1.y,
                      __uint_as_float(r[c * 8 + 6]) + b1.z, __uint_as_float(r[c * 8 + 7]) + b1.w};
        if (p.relu) {
#pragma unroll
          for (int q = 0; q < 8; ++q) v[q] = fmaxf(v[q], 0.f);
        }
        uint4 o;
        __half2* po = reinterpret_cast<__half2*>(&o);
#pragma unroll
        for (int q = 0; q < 4; ++q) po[q] = __floats2half2_rn(v[2 * q], v[2 * q + 1]);
        *reinterpret_cast<uint4*>(oslab + (((uint32_t)(chalf * 4 + c) ^ sw) << 4)) = o;
      }
      fence_proxy_async();
      named_bar_sync(1, 256);
      if (leader) {
        tma_store_4d(&p.out_map, out_stage + b * A_TILE_BYTES, 0, w0, h0, img);
        tma_store_commit();
      }
      if (++as == 2) {
        as = 0;
        aphase ^= 1u;
      }
    }
    if (leader) tma_store_wait<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<128>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------
// stem: conv 7x7 / 2, pad 3, 3 -> 64 (+ folded BN, optional ReLU) from NCHW fp32 to NHWC fp16
// (modelling/backbones/resnet.py:93-97,122-125 -- NO ReLU; resnet_ibn_a.py:84-86,126-129 -- ReLU)
// Direct convolution on the CUDA cores: K = 147 with Cin = 3 does not map on TMA channel slabs.
// Block: 8 x 32 output pixels x 64 channels, 256 threads, each 8 pixels (along w) x 8 channels.
// ---------------------------------------------------------------------------------------
static constexpr int ST_TH = 8, ST_TW = 32;
static constexpr int ST_PH = 2 * ST_TH + 5, ST_PW = 2 * ST_TW + 5;  // 21 x 69 input patch
static constexpr size_t STEM_SMEM = (size_t)(147 * 64 + 3 * ST_PH * (ST_PW + 1)) * sizeof(float);

__global__ void __launch_bounds__(256) stem_conv_kernel(const float* __restrict__ x, int H, int W,
                                                        const float* __restrict__ wt /*[147][64], k=(c*7+r)*7+s*/,
                                                        const float* __restrict__ bias, int relu,
                                                        __half* __restrict__ out, int Ho, int Wo) {
  extern __shared__ float ssm[];
  float* sw = ssm;                 // [147][64]
  float* sp = ssm + 147 * 64;      // [3][ST_PH][ST_PW + 1]
  const int n = blockIdx.z, oh0 = blockIdx.y * ST_TH, ow0 = blockIdx.x * ST_TW;
  for (int i = threadIdx.x; i < 147 * 64; i += 256) sw[i] = wt[i];
  const int ih0 = 2 * oh0 - 3, iw0 = 2 * ow0 - 3;
  for (int i = threadIdx.x; i < 3 * ST_PH * ST_PW; i += 256) {
    const int c = i / (ST_PH * ST_PW), rem = i % (ST_PH * ST_PW), ph = rem / ST_PW, pw = rem % ST_PW;
    const int ih = ih0 + ph, iw = iw0 + pw;
    float v = 0.f;
    if (ih >= 0 && ih < H && iw >= 0 && iw < W) v = x[(((size_t)n * 3 + c) * H + ih) * W + iw];
    sp[(c * ST_PH + ph) * (ST_PW + 1) + pw] = v;
  }
  __syncthreads();
  const int cg = threadIdx.x & 7;    // 8 channels
  const int pg = threadIdx.x >> 3;   // 32 pixel groups: row = pg / 4, 8 consecutive columns
  const int orow = pg >> 2, ocol0 = (pg & 3) * 8;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  for (int c = 0; c < 3; ++c)
    for (int r = 0; r < 7; ++r) {
      const float* prow = sp + (c * ST_PH + 2 * orow + r) * (ST_PW + 1) + 2 * ocol0;
#pragma unroll
      for (int s = 0; s < 7; ++s) {
        const float4 w0 = *reinterpret_cast<const float4*>(sw + ((c * 7 + r) * 7 + s) * 64 + cg * 8);
        const float4 w1 = *reinterpret_cast<const float4*>(sw + ((c * 7 + r) * 7 + s) * 64 + cg * 8 + 4);
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float xv = prow[2 * i + s];
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = __fmaf_rn(xv, wv[j], acc[i][j]);
        }
      }
    }
  const int oh = oh0 + orow;
  if (oh >= Ho) return;
  float b[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) b[j] = bias[cg * 8 + j];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ow = ow0 + ocol0 + i;
    if (ow >= Wo) continue;
    uint4 o;
    __half2* ph2 = reinterpret_cast<__half2*>(&o);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float a0 = acc[i][2 * j] + b[2 * j], a1 = acc[i][2 * j + 1] + b[2 * j + 1];
      if (relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); }
      ph2[j] = __floats2half2_rn(a0, a1);
    }
    *reinterpret_cast<uint4*>(out + (((size_t)n * Ho + oh) * Wo + ow) * 64 + cg * 8) = o;
  }
}

// ---------------------------------------------------------------------------------------
// stem on the tensor cores: the 7x7/2 convolution as a GEMM with K = 21 (c, r) groups x 8
// (s = 0..6 plus one zero column) = 168, padded to 192 = three 64-wide K slabs.
// Per tile of 4 x 32 output pixels: the fp32 NCHW input patch (13 x 72 x 3) is converted to
// fp16 in shared memory, every thread then assembles 16-byte K-chunks -- the 8 taps of one
// (c, r) group are 8 CONSECUTIVE patch columns -- straight into the SWIZZLE_128B operand
// layout (generic-proxy stores + fence.proxy.async), one thread issues 12 tcgen05.mma
// (M=128, N=64), and the epilogue adds the folded-BN bias (+ReLU for IBN) and writes one full
// 128-byte NHWC line per pixel.  Weights [64][192] fp16 stay resident in shared memory.
// ---------------------------------------------------------------------------------------
static constexpr int SK = 192;                    // padded K
static constexpr int S_TH = 4, S_TW = 32;         // output tile
static constexpr int S_PH = 2 * S_TH + 5;         // 13 input rows
static constexpr int S_PW = 72;                   // 2*32 + 5 = 69 input columns, padded to 72
static constexpr int STEM_BUILDERS = 256;                   // warps 0-7 assemble operand tiles
static constexpr int STEM_TC_THREADS = STEM_BUILDERS + 32 + 128;  // + MMA warp (8) + 4 epilogue warps (9-12)
static constexpr int S_A_BYTES = 3 * A_TILE_BYTES;          // 48 KiB: three [128][64] fp16 slabs
static constexpr int S_B_BYTES = 3 * 64 * 128;              // 24 KiB: three [64][64] fp16 slabs
static constexpr int S_PATCH_BYTES = 3 * S_PH * S_PW * 2;   // 5.6 KiB
static constexpr size_t STEM_TC_SMEM =
    2 * S_A_BYTES + S_B_BYTES + 2 * A_TILE_BYTES /*store staging*/ + 2 * S_PATCH_BYTES + 1024 + 128 + 256;

struct StemParams {
  CUtensorMap w_map;    // [64][192] fp16, box {64, 64}
  CUtensorMap out_map;  // NHWC fp16 output, box {64 ch, 32, 4, 1}
  const float* x;       // NCHW fp32
  const float* bias;
  __half* out;        // NHWC fp16 [n, Ho, Wo, 64]
  int n_img, H, W, Ho, Wo, tiles_h, tiles_w, relu;
};

// Persistent, one CTA per SM, three roles connected by mbarriers:
//   builders (8 warps): prefetched fp32 patch -> fp16 patch in smem -> swizzled operand tile A[buf]
//   MMA warp          : 12 tcgen05.mma (M=128, N=64) per tile into TMEM stage `as`
//   epilogue (4 warps): TMEM -> +bias (+ReLU) -> fp16 -> one 128-byte NHWC line per pixel
// A, the patch and the accumulator are double-buffered, so all three roles overlap.
__global__ void __launch_bounds__(STEM_TC_THREADS, 1) stem_tc_kernel(const __grid_constant__ StemParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sA = base, sB = base + 2 * S_A_BYTES, sO = sB + S_B_BYTES;
  constexpr int S_FIXED = 2 * S_A_BYTES + S_B_BYTES + 2 * A_TILE_BYTES;
  __half* patch0 = reinterpret_cast<__half*>(gbase + S_FIXED);
  const uint32_t bars = base + S_FIXED + 2 * S_PATCH_BYTES;
  const uint32_t bar_w = bars;  // weights landed
  auto a_full = [&](int b) { return bars + 8u * (1 + b); };
  auto a_empty = [&](int b) { return bars + 8u * (3 + b); };
  auto t_full = [&](int b) { return bars + 8u * (5 + b); };
  auto t_empty = [&](int b) { return bars + 8u * (7 + b); };
  const uint32_t tmem_slot = bars + 8u * 9;
  float* bias_s = reinterpret_cast<float*>(gbase + S_FIXED + 2 * S_PATCH_BYTES + 128);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid < 64) bias_s[tid] = p.bias[tid];
  if (tid == 0) {
    mbar_init(bar_w, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(a_full(b), STEM_BUILDERS / 32);  // one arrive per builder warp
      mbar_init(a_empty(b), 1);
      mbar_init(t_full(b), 1);
      mbar_init(t_empty(b), 4);
    }
    fence_barrier_init();
    tma_prefetch_desc(&p.w_map);
    tma_prefetch_desc(&p.out_map);
  }
  if (warp == 8) tmem_alloc<128>(tmem_slot);
  if (tid < STEM_BUILDERS) {
    // the three zero chunks (k = 168..191) of every pixel never change: chunks 5,6,7 of slab 2, both buffers
    for (int q = tid; q < 2 * 128 * 3; q += STEM_BUILDERS) {
      const int buf = q / 384, qq = q - buf * 384, px = qq & 127, ch = 5 + (qq >> 7);
      *reinterpret_cast<uint4*>(gbase + buf * S_A_BYTES + 2 * A_TILE_BYTES + px * 128 + ((ch ^ (px & 7)) << 4)) =
          make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();  // the next kernel may begin its prologue
  pdl_wait();               // activations of the previous kernel are complete and visible
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  const int tiles_per_img = p.tiles_h * p.tiles_w;
  const int num_tiles = p.n_img * tiles_per_img;

  if (tid < STEM_BUILDERS) {
    constexpr int NPRE = (3 * S_PH * S_PW + STEM_BUILDERS - 1) / STEM_BUILDERS;  // 11 loads in flight / thread
    float pre[NPRE];
    // tile-independent part of every patch element this thread owns: offset inside the image and (ph, pw)
    int p_off[NPRE], p_hw[NPRE];
#pragma unroll
    for (int j = 0; j < NPRE; ++j) {
      const int e = tid + j * STEM_BUILDERS;
      const int c = e / (S_PH * S_PW), rem = e - c * (S_PH * S_PW), ph = rem / S_PW, pw = rem - ph * S_PW;
      p_off[j] = (c * p.H + ph) * p.W + pw;
      p_hw[j] = e < 3 * S_PH * S_PW ? ((ph << 16) | pw) : (1 << 30);  // out-of-range marker fails the row test
    }
    auto load_patch = [&](int tile) {  // fp32 NCHW -> registers, zero outside the image
      const int img = tile / tiles_per_img, tr = tile - img * tiles_per_img;
      const int ih0 = 2 * ((tr / p.tiles_w) * S_TH) - 3, iw0 = 2 * ((tr % p.tiles_w) * S_TW) - 3;
      const float* xb = p.x + (size_t)img * 3 * p.H * p.W + (long long)ih0 * p.W + iw0;
#pragma unroll
      for (int j = 0; j < NPRE; ++j) {
        const int ih = ih0 + (p_hw[j] >> 16), iw = iw0 + (p_hw[j] & 0xFFFF);
        float v = 0.f;
        if ((unsigned)ih < (unsigned)p.H && (unsigned)iw < (unsigned)p.W) v = __ldg(xb + p_off[j]);
        pre[j] = v;
      }
    };
    // per-thread constants of the operand assembly: pixel px, (c, r) groups cr = 2 i + hi
    const int px = tid & 127, hi = tid >> 7;
    int src_off[11], dst_off[11];
#pragma unroll
    for (int i = 0; i < 11; ++i) {
      const int cr = 2 * i + hi, c = cr / 7, r = cr - c * 7;
      src_off[i] = (c * S_PH + 2 * (px >> 5) + r) * S_PW + 2 * (px & 31);
      dst_off[i] = (cr >> 3) * A_TILE_BYTES + px * 128 + (((cr & 7) ^ (px & 7)) << 4);
    }
    if ((int)blockIdx.x < num_tiles) load_patch(blockIdx.x);
    int buf = 0;
    uint32_t eph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      __half* patch = patch0 + buf * (S_PATCH_BYTES / 2);
#pragma unroll
      for (int j = 0; j < NPRE; ++j) {
        const int e = tid + j * STEM_BUILDERS;
        if (e < 3 * S_PH * S_PW) patch[e] = __float2half_rn(pre[j]);
      }
      named_bar_sync(2, STEM_BUILDERS);  // patch[buf] complete (its previous readers finished two tiles ago)
      if (tile + (int)gridDim.x < num_tiles) load_patch(tile + gridDim.x);  // next patch travels during the build
      mbar_wait(a_empty(buf), eph ^ 1u);  // the MMAs that read A[buf] two tiles ago have completed
      uint8_t* A = gbase + buf * S_A_BYTES;
#pragma unroll
      for (int i = 0; i < 11; ++i) {
        if (2 * i + hi < 21) {
          const uint32_t* src = reinterpret_cast<const uint32_t*>(patch + src_off[i]);
          *reinterpret_cast<uint4*>(A + dst_off[i]) = make_uint4(src[0], src[1], src[2], src[3]);
        }
      }
      fence_proxy_async();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full(buf));
      if (++buf == 2) {
        buf = 0;
        eph ^= 1u;
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      mbar_arrive_expect_tx(bar_w, S_B_BYTES);
      for (int kb = 0; kb < 3; ++kb) tma_load_2d(sB + kb * 64 * 128, &p.w_map, bar_w, kb * 64, 0);
      mbar_wait(bar_w, 0);
      constexpr uint32_t idesc = make_idesc_f16(128, 64);
      int buf = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(t_empty(buf), ph ^ 1u);  // accumulator stage drained
        mbar_wait(a_full(buf), ph);        // operand tile assembled
        tc_fence_after();
#pragma unroll
        for (int kb = 0; kb < 3; ++kb) {
          const uint64_t da = make_sw128_kmajor_desc(sA + buf * S_A_BYTES + kb * A_TILE_BYTES);
          const uint64_t db = make_sw128_kmajor_desc(sB + kb * 64 * 128);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16(tmem_base + buf * 64, desc_advance_k(da, k), desc_advance_k(db, k), idesc, (kb | k) ? 1u : 0u);
        }
        umma_commit(a_empty(buf));
        umma_commit(t_full(buf));
        if (++buf == 2) {
          buf = 0;
          ph ^= 1u;
        }
      }
    }
  } else {
    const int quarter = warp & 3;  // warps 9..12 -> quarters 1,2,3,0
    const int px = quarter * 32 + lane;
    const bool leader = (warp == 9 && lane == 0);
    int buf = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int img = tile / tiles_per_img, tr = tile - img * tiles_per_img;
      const int oh0 = (tr / p.tiles_w) * S_TH, ow0 = (tr % p.tiles_w) * S_TW;
      mbar_wait(t_full(buf), ph);
      tc_fence_after();
      uint32_t r[64];
      const uint32_t t0 = tmem_base + buf * 64 + (static_cast<uint32_t>(quarter * 32) << 16);
      tmem_ld16(t0, *reinterpret_cast<uint32_t(*)[16]>(&r[0]));
      tmem_ld16(t0 + 16, *reinterpret_cast<uint32_t(*)[16]>(&r[16]));
      tmem_ld16(t0 + 32, *reinterpret_cast<uint32_t(*)[16]>(&r[32]));
      tmem_ld16(t0 + 48, *reinterpret_cast<uint32_t(*)[16]>(&r[48]));
      if (leader) tma_store_wait_read<1>();  // staging slab `buf` was stored two tiles ago
      named_bar_sync(3, 128);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(t_empty(buf));
      uint8_t* slab = gbase + 2 * S_A_BYTES + S_B_BYTES + buf * A_TILE_BYTES + px * 128;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        uint4 o;
        __half2* po = reinterpret_cast<__half2*>(&o);
        const float4 bA = *reinterpret_cast<const float4*>(bias_s + c * 8);
        const float4 bB = *reinterpret_cast<const float4*>(bias_s + c * 8 + 4);
        const float bv[8] = {bA.x, bA.y, bA.z, bA.w, bB.x, bB.y, bB.z, bB.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float a0 = __uint_as_float(r[c * 8 + 2 * q]) + bv[2 * q];
          float a1 = __uint_as_float(r[c * 8 + 2 * q + 1]) + bv[2 * q + 1];
          if (p.relu) {
            a0 = fmaxf(a0, 0.f);
            a1 = fmaxf(a1, 0.f);
          }
          po[q] = __floats2half2_rn(a0, a1);
        }
        *reinterpret_cast<uint4*>(slab + ((c ^ (px & 7)) << 4)) = o;
      }
      fence_proxy_async();
      named_bar_sync(3, 128);
      if (leader) {
        tma_store_4d(&p.out_map, sO + buf * A_TILE_BYTES, 0, ow0, oh0, img);
        tma_store_commit();
      }
      if (++buf == 2) {
        buf = 0;
        ph ^= 1u;
      }
    }
    if (leader) tma_store_wait<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<128>(tmem_base);
  }
}

// =======================================================================================
// Fused stem: conv 7x7 / 2 (+folded BN, optional ReLU) -> maxpool 3x3 / 2, for inputs up to 128 pixels wide.
//
// The input is first packed to zero-bordered NHWC4 fp16 (stem_pack_input_kernel: [N][H+6][136][4], 8 bytes per
// pixel, 3 border pixels left/top).  In that layout the 7-pixel window of output column ox starts 16 bytes after
// the window of ox-1 (stride 2 x 8 bytes), which is exactly the row pitch of a K-major NO-SWIZZLE UMMA core
// matrix (8 rows, 16 bytes apart).  So the im2col operand is never built: shared memory holds raw input rows
// (cut into 8 overlapping 192-byte pieces of 8 output columns each by one TMA box with overlapping strides) and
// the A descriptor (LBO = 16 B, SBO = 192 B) walks the windows in place.  Per output-row pair the CTA loads
// 10 input-row slots (15 KiB) instead of a 56 KiB im2col tile; K = 7 kernel rows x (8 px x 4 ch) = 224.
// Even/odd input rows sit in separate slot runs so that "+1 slot" = "+2 input rows" = the second output row
// (rows 64..127 of the M = 128 tile).
//
// The epilogue writes the conv tile (2 output rows x 64 columns x 64 ch, fp16) to a triple-buffered smem tile and
// pools it together with the last row of the previous tile; only the pooled tensor goes to HBM.  A CTA walks a
// contiguous range of row pairs; a range that starts inside an image first recomputes the row pair above it.
// =======================================================================================
static constexpr int S3_THREADS = 448;                 // TMA warp, MMA warp, 8 epilogue warps, 4 pool warps
static constexpr int S3_STAGES = 4;
static constexpr int S3_PIECE = 256;                   // bytes: 8 windows (stride 2 px) of 8 px need 176; 256 keeps core matrices 128 B-aligned
static constexpr int S3_SLOT = 8 * S3_PIECE;           // one input row cut into 8 pieces
static constexpr int S3_STAGE_BYTES = 10 * S3_SLOT;    // 5 even + 5 odd input rows
static constexpr int S3_W_BYTES = 28 * 64 * 16;        // [k chunk of 8][cout][8] fp16
static constexpr int S3_TILE_BYTES = 128 * 128;        // conv tile, one 128-byte line per pixel
static constexpr int S3_WP = 136;                      // padded input row, pixels
static constexpr size_t S3_SMEM = 1024 + S3_STAGES * S3_STAGE_BYTES + S3_W_BYTES + 3 * S3_TILE_BYTES + 256 + 256;

struct Stem3Params {
  CUtensorMap x_map;  // 5-D overlapping view of the packed input: {96 el, 8 pieces, row pair, parity, image}
  const __half* w;    // packed weights [28][64][8]
  const float* bias;
  __half* out;        // pooled NHWC fp16 [n][hp][wp][64]
  int n_img, hp, wp, Wo, relu;
};

// NCHW fp32 -> zero-bordered NHWC4 fp16; block = 64 x 4 threads, a thread converts two adjacent pixels of one row
__global__ void __launch_bounds__(256) stem_pack_input_kernel(const float* __restrict__ x, int N, int H, int W,
                                                              __half* __restrict__ xp) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x * 4 + (threadIdx.x >> 6);  // n * H + y
  const int xw = 2 * (threadIdx.x & 63);
  if (row >= N * H || xw >= W) return;
  const int n = row / H, y = row - n * H;
  const size_t plane = (size_t)H * W;
  const float* src = x + (size_t)n * 3 * plane + (size_t)y * W + xw;
  const float2 c0 = *reinterpret_cast<const float2*>(src);
  const float2 c1 = *reinterpret_cast<const float2*>(src + plane);
  const float2 c2 = *reinterpret_cast<const float2*>(src + 2 * plane);
  const __half2 a0 = __floats2half2_rn(c0.x, c1.x), b0 = __floats2half2_rn(c2.x, 0.f);
  const __half2 a1 = __floats2half2_rn(c0.y, c1.y), b1 = __floats2half2_rn(c2.y, 0.f);
  uint2* dst = reinterpret_cast<uint2*>(xp + (((size_t)n * (H + 6) + y + 3) * S3_WP + xw + 3) * 4);
  dst[0] = make_uint2(*reinterpret_cast<const uint32_t*>(&a0), *reinterpret_cast<const uint32_t*>(&b0));
  dst[1] = make_uint2(*reinterpret_cast<const uint32_t*>(&a1), *reinterpret_cast<const uint32_t*>(&b1));
}

// The same packed layout straight from uint8 HWC crops: ToTensor + Normalize (datasets/transforms/build.py:29-33) folded
// into the pack -- (u / 255 - mean) / std in IEEE fp32 (the arithmetic of augment_kernel, so the fp16 operand is
// bit-identical to normalize_batch followed by stem_pack_input_kernel) without the fp32 NCHW tensor in between
// (3 B read per pixel instead of 12 B written + 12 B read).
__global__ void __launch_bounds__(256) stem_pack_input_u8_kernel(const uint8_t* __restrict__ x, int N, int H, int W, float m0,
                                                                 float m1, float m2, float s0, float s1, float s2,
                                                                 __half* __restrict__ xp) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x * 4 + (threadIdx.x >> 6);  // n * H + y
  const int xw = 2 * (threadIdx.x & 63);
  if (row >= N * H || xw >= W) return;
  const int n = row / H, y = row - n * H;
  const uint16_t* src = reinterpret_cast<const uint16_t*>(x + ((size_t)row * W + xw) * 3);  // 6 bytes, 2-byte aligned
  const uint32_t w0 = src[0], w1 = src[1], w2 = src[2];  // r0 g0 | b0 r1 | g1 b1
  const float r0 = (float)(w0 & 255u) / 255.f, g0 = (float)(w0 >> 8) / 255.f, b0 = (float)(w1 & 255u) / 255.f;
  const float r1 = (float)(w1 >> 8) / 255.f, g1 = (float)(w2 & 255u) / 255.f, b1 = (float)(w2 >> 8) / 255.f;
  const __half2 a0 = __floats2half2_rn((r0 - m0) / s0, (g0 - m1) / s1), c0 = __floats2half2_rn((b0 - m2) / s2, 0.f);
  const __half2 a1 = __floats2half2_rn((r1 - m0) / s0, (g1 - m1) / s1), c1 = __floats2half2_rn((b1 - m2) / s2, 0.f);
  uint2* dst = reinterpret_cast<uint2*>(xp + (((size_t)n * (H + 6) + y + 3) * S3_WP + xw + 3) * 4);
  dst[0] = make_uint2(*reinterpret_cast<const uint32_t*>(&a0), *reinterpret_cast<const uint32_t*>(&c0));
  dst[1] = make_uint2(*reinterpret_cast<const uint32_t*>(&a1), *reinterpret_cast<const uint32_t*>(&c1));
}

__global__ void __launch_bounds__(S3_THREADS, 1) stem_pool_kernel(const __grid_constant__ Stem3Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t sA = base, sW = sA + S3_STAGES * S3_STAGE_BYTES, sT = sW + S3_W_BYTES;
  uint8_t* tile_g = gbase + (sT - base);
  float* bias_s = reinterpret_cast<float*>(gbase + (sT - base) + 3 * S3_TILE_BYTES);
  const uint32_t bars = sT + 3 * S3_TILE_BYTES + 256;
  const uint32_t bar_w = bars;
  auto full_bar = [&](int s) { return bars + 8u * (1 + s); };
  auto empty_bar = [&](int s) { return bars + 8u * (1 + S3_STAGES + s); };
  auto tfull_bar = [&](int s) { return bars + 8u * (1 + 2 * S3_STAGES + s); };
  auto tempty_bar = [&](int s) { return bars + 8u * (3 + 2 * S3_STAGES + s); };
  auto sfull_bar = [&](int s) { return bars + 8u * (5 + 2 * S3_STAGES + s); };   // conv tile written (8 warps)
  auto sempty_bar = [&](int s) { return bars + 8u * (8 + 2 * S3_STAGES + s); };  // conv tile no longer needed (4 warps)
  const uint32_t tmem_slot = bars + 8u * (11 + 2 * S3_STAGES);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid < 64) bias_s[tid] = p.bias[tid];
  if (tid == 0) {
    mbar_init(bar_w, 1);
    for (int s = 0; s < S3_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 8);
    }
    for (int s = 0; s < 3; ++s) {
      mbar_init(sfull_bar(s), 8);
      mbar_init(sempty_bar(s), 4);
    }
    fence_barrier_init();
    tma_prefetch_desc(&p.x_map);
  }
  if (warp == 1) tmem_alloc<128>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  // contiguous, balanced range of row pairs; a range that starts inside an image recomputes the pair above it
  const int num_tiles = p.n_img * p.hp;
  const int per = num_tiles / (int)gridDim.x, rem = num_tiles - per * (int)gridDim.x;
  const int t_begin = (int)blockIdx.x * per + min((int)blockIdx.x, rem);
  const int t_end = t_begin + per + ((int)blockIdx.x < rem ? 1 : 0);
  const int t_first = (t_begin < t_end && (t_begin % p.hp) != 0) ? t_begin - 1 : t_begin;

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(bar_w, S3_W_BYTES);
      bulk_copy_g2s(sW, p.w, S3_W_BYTES, bar_w);
      int stage = 0;
      uint32_t phase = 0;
      for (int t = t_first; t < t_end; ++t) {
        const int n = t / p.hp, py = t - n * p.hp;
        mbar_wait(empty_bar(stage), phase ^ 1u);
        const uint32_t dst = sA + stage * S3_STAGE_BYTES;
        mbar_arrive_expect_tx(full_bar(stage), S3_STAGE_BYTES);
        tma_load_5d(dst, &p.x_map, full_bar(stage), 0, 0, 2 * py, 0, n);                   // padded rows 4py, +2, .., +8
        tma_load_5d(dst + 5 * S3_SLOT, &p.x_map, full_bar(stage), 0, 0, 2 * py, 1, n);     // padded rows 4py+1, .., +9
        if (++stage == S3_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(128, 64);
      mbar_wait(bar_w, 0);
      tc_fence_after();
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      for (int t = t_first; t < t_end; ++t) {
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        mbar_wait(full_bar(stage), phase);
        tc_fence_after();
        const uint32_t a0 = sA + stage * S3_STAGE_BYTES;
        const uint32_t acc = tmem_base + as * 64;
#pragma unroll
        for (int r = 0; r < 7; ++r) {
          // kernel row r of output row 0 = padded input row 4py + r: slot r/2 of the even or odd run; rows 64..127
          // of the tile (output row 1) land one slot further (SBO * 8 = one slot)
          const uint32_t arow = a0 + ((r & 1) * 5 + (r >> 1)) * S3_SLOT;
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            const uint64_t da = make_noswizzle_kmajor_desc(arow + 32 * kk, 16, S3_PIECE);
            const uint64_t db = make_noswizzle_kmajor_desc(sW + (r * 4 + 2 * kk) * 1024, 1024, 128);
            umma_f16(acc, da, db, idesc, (r > 0 || kk > 0) ? 1u : 0u);
          }
        }
        umma_commit(empty_bar(stage));
        umma_commit(tfull_bar(as));
        if (++stage == S3_STAGES) {
          stage = 0;
          phase ^= 1u;
        }
        if (++as == 2) {
          as = 0;
          aphase ^= 1u;
        }
      }
    }
  } else if (warp < 10) {
    // ---- epilogue warps: TMEM -> +bias (+ReLU) -> fp16 -> conv tile in shared memory (ring of 3) ----
    const int ew = warp - 2;
    const int quarter = warp & 3, chalf = ew >> 2;
    const int px = quarter * 32 + lane;  // tile row: output row px / 64, column px % 64
    int as = 0, buf = 0;
    uint32_t aphase = 0, bphase = 0;
    float bs[32];  // this thread's 32 channels never change: bias lives in registers (no per-tile LDS)
#pragma unroll
    for (int j = 0; j < 32; ++j) bs[j] = bias_s[chalf * 32 + j];
    for (int t = t_first; t < t_end; ++t) {
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      uint32_t r0[16], r1[16];
      const uint32_t taddr = tmem_base + as * 64 + chalf * 32 + (static_cast<uint32_t>(quarter * 32) << 16);
      tmem_ld16(taddr, r0);
      tmem_ld16(taddr + 16, r1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(as));
      uint8_t* tl = tile_g + buf * S3_TILE_BYTES;
      uint32_t h[16];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float v0 = __uint_as_float(r0[2 * j]) + bs[2 * j], v1 = __uint_as_float(r0[2 * j + 1]) + bs[2 * j + 1];
        float v2 = __uint_as_float(r1[2 * j]) + bs[16 + 2 * j], v3 = __uint_as_float(r1[2 * j + 1]) + bs[16 + 2 * j + 1];
        if (p.relu) {
          v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f);
        }
        const __half2 a = __floats2half2_rn(v0, v1), b = __floats2half2_rn(v2, v3);
        h[j] = *reinterpret_cast<const uint32_t*>(&a);
        h[8 + j] = *reinterpret_cast<const uint32_t*>(&b);
      }
      mbar_wait(sempty_bar(buf), bphase ^ 1u);  // the pool warps are done with the tile that lived here
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int chunk = chalf * 4 + q;
        *reinterpret_cast<uint4*>(tl + px * 128 + ((chunk ^ (px & 7)) << 4)) =
            make_uint4(h[4 * q], h[4 * q + 1], h[4 * q + 2], h[4 * q + 3]);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(sfull_bar(buf));
      if (++buf == 3) {
        buf = 0;
        bphase ^= 1u;
      }
      if (++as == 2) {
        as = 0;
        aphase ^= 1u;
      }
    }
  } else {
    // ---- pool warps: 3x3/2 max over the conv tile and the last row of the previous one -> HBM ----
    const int pt = tid - 320;  // 0..127
    int buf = 0;
    uint32_t bphase = 0;
    for (int t = t_first; t < t_end; ++t) {
      const int n = t / p.hp, py = t - n * p.hp;
      mbar_wait(sfull_bar(buf), bphase);
      const int pbuf = buf == 0 ? 2 : buf - 1;
      if (t >= t_begin) {
        const uint8_t* tl = tile_g + buf * S3_TILE_BYTES;
        const uint8_t* prev = tile_g + pbuf * S3_TILE_BYTES;
        // Out-of-range taps are replaced by an in-window duplicate (max is idempotent): all 9 loads of an output are
        // unconditional and issued back to back (one shared-memory round trip, not nine).
        const uint8_t* rows[3] = {py == 0 ? tl : prev + 64 * 128, tl, tl + 64 * 128};
#pragma unroll
        for (int it = 0; it < 2; ++it) {
          const int item = pt + it * 128;
          const int ppx = min(item >> 3, p.wp - 1), pch = item & 7;  // pooled column, 8-channel chunk
          const int cxs[3] = {max(2 * ppx - 1, 0), 2 * ppx, min(2 * ppx + 1, p.Wo - 1)};
          uint4 v[9];
#pragma unroll
          for (int dy = 0; dy < 3; ++dy)
#pragma unroll
            for (int dx = 0; dx < 3; ++dx)
              v[dy * 3 + dx] = *reinterpret_cast<const uint4*>(rows[dy] + cxs[dx] * 128 + ((pch ^ (cxs[dx] & 7)) << 4));
          uint4 m = v[0];
          __half2* mm = reinterpret_cast<__half2*>(&m);
#pragma unroll
          for (int q = 1; q < 9; ++q) {
            const __half2* vv = reinterpret_cast<const __half2*>(&v[q]);
#pragma unroll
            for (int e = 0; e < 4; ++e) mm[e] = __hmax2(mm[e], vv[e]);
          }
          if ((item >> 3) < p.wp)
            *reinterpret_cast<uint4*>(p.out + (((size_t)n * p.hp + py) * p.wp + ppx) * 64 + pch * 8) = m;
        }
      }
      __syncwarp();
      if (lane == 0 && t > t_first) mbar_arrive(sempty_bar(pbuf));  // the previous tile is no longer needed
      if (++buf == 3) {
        buf = 0;
        bphase ^= 1u;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc<128>(tmem_base);
  }
}

// maxpool 3x3 / 2, pad 1, NHWC fp16; one thread = 8 channels of one output pixel
__global__ void __launch_bounds__(256) maxpool3x3s2_kernel(const __half* __restrict__ x, int N, int H, int W, int C,
                                                           __half* __restrict__ out, int Ho, int Wo) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int cv = C / 8;
  const size_t total = (size_t)N * Ho * Wo * cv;
  if (i >= total) return;
  const int c8 = (int)(i % cv);
  size_t t = i / cv;
  const int ow = (int)(t % Wo);
  t /= Wo;
  const int oh = (int)(t % Ho);
  const int n = (int)(t / Ho);
  __half2 m[4];
  const __half2 neg = __float2half2_rn(-65504.f);
#pragma unroll
  for (int j = 0; j < 4; ++j) m[j] = neg;
  for (int r = 0; r < 3; ++r) {
    const int ih = 2 * oh - 1 + r;
    if (ih < 0 || ih >= H) continue;
    for (int s = 0; s < 3; ++s) {
      const int iw = 2 * ow - 1 + s;
      if (iw < 0 || iw >= W) continue;
      const uint4 v = *reinterpret_cast<const uint4*>(x + (((size_t)n * H + ih) * W + iw) * C + c8 * 8);
      const __half2* hv = reinterpret_cast<const __half2*>(&v);
#pragma unroll
      for (int j = 0; j < 4; ++j) m[j] = __hmax2(m[j], hv[j]);
    }
  }
  uint4 o;
  __half2* po = reinterpret_cast<__half2*>(&o);
#pragma unroll
  for (int j = 0; j < 4; ++j) po[j] = m[j];
  *reinterpret_cast<uint4*>(out + (((size_t)n * Ho + oh) * Wo + ow) * C + c8 * 8) = o;
}

// global average pool over H*W (fp32 accumulate, pixel order) + optional eval BatchNorm1d
// (modelling/baseline.py:93-94, modelling/bases.py:175): one thread = 2 channels of one image
__global__ void __launch_bounds__(256) gap_bn_kernel(const __half* __restrict__ x, int HW, int C,
                                                     const float* __restrict__ bn_scale /*gamma/sqrt(var+eps)*/,
                                                     const float* __restrict__ bn_shift, float* __restrict__ feat,
                                                     float* __restrict__ emb) {
  pdl_launch_dependents();
  pdl_wait();
  const int n = blockIdx.y;
  const int c2 = blockIdx.x * blockDim.x + threadIdx.x;
  if (c2 * 2 >= C) return;
  const __half2* base = reinterpret_cast<const __half2*>(x + (size_t)n * HW * C) + c2;
  float s0 = 0.f, s1 = 0.f;
  for (int p = 0; p < HW; ++p) {
    const float2 v = __half22float2(base[(size_t)p * (C / 2)]);
    s0 += v.x;
    s1 += v.y;
  }
  const float inv = 1.f / (float)HW;
  const float f0 = s0 * inv, f1 = s1 * inv;
  if (feat) {
    feat[(size_t)n * C + 2 * c2] = f0;
    feat[(size_t)n * C + 2 * c2 + 1] = f1;
  }
  if (emb) {
    emb[(size_t)n * C + 2 * c2] = __fmaf_rn(f0, bn_scale[2 * c2], bn_shift[2 * c2]);
    emb[(size_t)n * C + 2 * c2 + 1] = __fmaf_rn(f1, bn_scale[2 * c2 + 1], bn_shift[2 * c2 + 1]);
  }
}

// InstanceNorm2d(affine, instance statistics) + ReLU in place on channels [0, half) of an NHWC
// fp16 tensor (IBN, resnet_ibn_a.py:18-32): one block per (image, 8-channel group).
__global__ void __launch_bounds__(256) instnorm_relu_kernel(__half* __restrict__ x, int HW, int C, int half,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s_sum[8][8], s_sq[8][8];
  __shared__ float s_mean[8], s_istd[8];
  const int n = blockIdx.y, c0 = blockIdx.x * 8;
  if (c0 >= half) return;
  __half* base = x + (size_t)n * HW * C + c0;
  float s[8] = {}, q[8] = {};
  for (int p = threadIdx.x; p < HW; p += blockDim.x) {
    const uint4 v = *reinterpret_cast<const uint4*>(base + (size_t)p * C);
    const __half2* hv = reinterpret_cast<const __half2*>(&v);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(hv[j]);
      s[2 * j] += f.x; q[2 * j] = __fmaf_rn(f.x, f.x, q[2 * j]);
      s[2 * j + 1] += f.y; q[2 * j + 1] = __fmaf_rn(f.y, f.y, q[2 * j + 1]);
    }
  }
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
      q[j] += __shfl_xor_sync(0xffffffffu, q[j], o);
    }
    if (lane == 0) { s_sum[wp][j] = s[j]; s_sq[wp][j] = q[j]; }
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    float ts = 0.f, tq = 0.f;
    for (int w = 0; w < 8; ++w) { ts += s_sum[w][threadIdx.x]; tq += s_sq[w][threadIdx.x]; }
    const float mean = ts / (float)HW;
    const float var = fmaxf(tq / (float)HW - mean * mean, 0.f);  // biased, like F.instance_norm
    s_mean[threadIdx.x] = mean;
    s_istd[threadIdx.x] = rsqrtf(var + eps);
  }
  __syncthreads();
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = gamma[c0 + j] * s_istd[j];
    sh[j] = beta[c0 + j] - s_mean[j] * sc[j];
  }
  for (int p = threadIdx.x; p < HW; p += blockDim.x) {
    uint4 v = *reinterpret_cast<const uint4*>(base + (size_t)p * C);
    __half2* hv = reinterpret_cast<__half2*>(&v);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(hv[j]);
      hv[j] = __floats2half2_rn(fmaxf(__fmaf_rn(f.x, sc[2 * j], sh[2 * j]), 0.f),
                                fmaxf(__fmaf_rn(f.y, sc[2 * j + 1], sh[2 * j + 1]), 0.f));
    }
    *reinterpret_cast<uint4*>(base + (size_t)p * C) = v;
  }
}

// ---------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------
template <int BN>
static int launch_conv(const ConvKernelParams& p, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    CTL_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)ConvCfg<BN>::SMEM));
    attr_set = true;
  }
  const long long tiles = (long long)p.m_tiles * p.n_tiles;
  const int grid = (int)std::min<long long>(tiles, sm_count());
  CTL_CUDA(launch_k(conv_gemm_kernel<BN>, dim3(grid), dim3(CONV_THREADS), ConvCfg<BN>::SMEM, st, p));
  CTL_LAUNCH_CHECK();
  return 0;
}

static int launch_c64(const void* x, int n, int h, int w, const void* weight, const float* bias, void* out, int relu,
                      cudaStream_t st) {
  C64Params p = {};
  p.bias = bias;
  p.n_img = n;
  p.H = h;
  p.W = w;
  p.tiles_h = (h + 15) / 16;
  p.tiles_w = (w + 7) / 8;
  p.relu = relu;
  p.use_base_offset = 0;  // see the kernel comment: shifted views need no base_offset
  int rc;
  const uint64_t dims[4] = {64, (uint64_t)w, (uint64_t)h, (uint64_t)n};
  const uint64_t strd[4] = {2, 128, (uint64_t)w * 128, (uint64_t)h * w * 128};
  const uint32_t xbox[4] = {64, 16, 18, 1}, obox[4] = {64, 8, 16, 1};
  if ((rc = encode_tensor_map(&p.x_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 4, x, dims, strd, xbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = encode_tensor_map(&p.out_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 4, out, dims, strd, obox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  const uint64_t wd[2] = {576, 64}, ws[2] = {2, 576 * 2};
  const uint32_t wbox[2] = {64, 64};
  if ((rc = encode_tensor_map(&p.w_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 2, weight, wd, ws, wbox, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    CTL_CUDA(cudaFuncSetAttribute(conv3x3_c64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C64_SMEM));
    attr_set = true;
  }
  const long long tiles = (long long)n * p.tiles_h * p.tiles_w;
  const int grid = (int)std::min<long long>(tiles, sm_count());
  CTL_CUDA(launch_k(conv3x3_c64_kernel, dim3(grid), dim3(CONV_THREADS), C64_SMEM, st, p));
  CTL_LAUNCH_CHECK();
  return 0;
}

template <int BN, int VAR>
static int launch_conv_pair_v(const ConvKernelParams& p, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    CTL_CUDA(cudaFuncSetAttribute(conv_gemm_pair_kernel<BN, VAR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)PairCfg<BN, VAR>::SMEM));
    attr_set = true;
  }
  const long long tiles = (long long)(p.m_tiles / 2) * p.n_tiles;
  const int clusters = (int)std::min<long long>(tiles, sm_count() / 2);
  CTL_CUDA(launch_k(conv_gemm_pair_kernel<BN, VAR>, dim3(2 * clusters), dim3(CONV_THREADS), PairCfg<BN, VAR>::SMEM, st, p));
  CTL_LAUNCH_CHECK();
  return 0;
}

template <int BN>
static int launch_conv_pair(const ConvKernelParams& p, cudaStream_t st) {
  return p.has_residual ? launch_conv_pair_v<BN, 2>(p, st) : launch_conv_pair_v<BN, 1>(p, st);
}

// Fills the tile geometry, the output / residual / weight maps and dispatches.  The caller has filled the A maps,
// the taps and k_blocks; `ktot` = row length of the weight matrix [Cout][ktot].
static int finish_and_launch(ConvKernelParams& p, int n, int Ho, int Wo, int cout, int ktot, const void* weight,
                             const float* bias, const void* residual, void* out, int relu, int relu_from,
                             cudaStream_t st) {
  int rc;
  p.n_img = n;
  p.Ho = Ho;
  p.Wo = Wo;
  p.Cout = cout;
  p.bias = bias;
  p.has_residual = residual != nullptr;
  p.relu = relu;
  p.relu_from = relu_from;
  p.m_tiles = n * p.tiles_h * p.tiles_w;
  const int BN = cout % 256 == 0 ? 256 : (cout % 128 == 0 ? 128 : 64);
  p.n_tiles = cout / BN;
  {
    const uint64_t odims[4] = {(uint64_t)cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)n};
    const uint64_t ostr[4] = {2, (uint64_t)cout * 2, (uint64_t)Wo * cout * 2, (uint64_t)Ho * Wo * cout * 2};
    const uint32_t obox[4] = {64, (uint32_t)p.TW, (uint32_t)p.TH, 1};
    if ((rc = encode_tensor_map(&p.out_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 4, out, odims, ostr, obox,
                                CU_TENSOR_MAP_SWIZZLE_128B)))
      return rc;
    if ((rc = encode_tensor_map(&p.res_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 4, residual ? residual : out, odims,
                                ostr, obox, CU_TENSOR_MAP_SWIZZLE_128B)))
      return rc;
  }
  // CTA pairs for every 256- / 128-channel-tile layer with an even tile count; CTL_CONV_PAIR=0 forces the single-CTA
  // kernel (A/B runs)
  static const int pair_mode = [] { const char* e = getenv("CTL_CONV_PAIR"); return e ? atoi(e) : -1; }();
  const bool use_pair = (BN == 256 || BN == 128) && (p.m_tiles % 2 == 0) && p.m_tiles >= 2 && pair_mode != 0;
  const uint64_t bdims[2] = {(uint64_t)ktot, (uint64_t)cout};
  const uint64_t bstr[2] = {2, (uint64_t)ktot * 2};
  const uint32_t bbox[2] = {CBK, (uint32_t)(use_pair ? BN / 2 : BN)};  // a pair CTA stages half of the weight tile
  if ((rc = encode_tensor_map(&p.b_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 2, weight, bdims, bstr, bbox,
                              CU_TENSOR_MAP_SWIZZLE_128B)))
    return rc;
  if (use_pair) return BN == 256 ? launch_conv_pair<256>(p, st) : launch_conv_pair<128>(p, st);
  if (BN == 256) return launch_conv<256>(p, st);
  if (BN == 128) return launch_conv<128>(p, st);
  return launch_conv<64>(p, st);
}

// rows (columns) of a side of `size` pixels whose index has parity `parity`: the extent of a stride-2 parity view
static inline int parity_extent(int size, int parity) { return (size - parity + 1) / 2; }

// A tensor maps of one NHWC source [n, h, w, cin] read at `stride`: stride 1 -> map 0..3 identical; stride 2 -> the four
// parity views (view (ph, pw) holds input pixels (2i + ph, 2j + pw)), so every box is a dense stride-1 box.  Each view
// has its own extent parity_extent(h, ph) x parity_extent(w, pw): on an odd side the odd view is one pixel shorter, and
// the TMA zero-fill past its end is the convolution's zero padding.  A view that is empty (h == 1 or w == 1) gets a copy
// of view (0, 0) so that every descriptor is valid; the caller issues no tap on it.
static int encode_source(CUtensorMap* maps, int count, const void* x, int n, int h, int w, int cin, int stride, int TH,
                         int TW) {
  int rc;
  const __half* xb = static_cast<const __half*>(x);
  const uint32_t abox[4] = {CBK, (uint32_t)TW, (uint32_t)TH, 1};
  if (stride == 1) {
    const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)w, (uint64_t)h, (uint64_t)n};
    const uint64_t strd[4] = {2, (uint64_t)cin * 2, (uint64_t)w * cin * 2, (uint64_t)h * w * cin * 2};
    for (int i = 0; i < count; ++i)
      if ((rc = encode_tensor_map(&maps[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 4, xb, dims, strd, abox,
                                  CU_TENSOR_MAP_SWIZZLE_128B)))
        return rc;
    return 0;
  }
  const uint64_t strd[4] = {2, (uint64_t)cin * 4, (uint64_t)w * cin * 4, (uint64_t)h * w * cin * 2};
  for (int v = 0; v < count; ++v) {
    const int ph = v >> 1, pw = v & 1;
    const int vh = parity_extent(h, ph), vw = parity_extent(w, pw);
    if (vh == 0 || vw == 0) {
      maps[v] = maps[0];
      continue;
    }
    const uint64_t dims[4] = {(uint64_t)cin, (uint64_t)vw, (uint64_t)vh, (uint64_t)n};
    if ((rc = encode_tensor_map(&maps[v], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 4, xb + ((size_t)ph * w + pw) * cin, dims,
                                strd, abox, CU_TENSOR_MAP_SWIZZLE_128B)))
      return rc;
  }
  return 0;
}

}  // namespace ctl

using namespace ctl;

extern "C" {

int ctl_conv2d_nhwc_f16(const void* x, int32_t n, int32_t h, int32_t w, int32_t cin, const void* weight,
                        const float* bias, const void* residual, void* out, int32_t cout, int32_t ksize,
                        int32_t stride, int32_t relu, int32_t relu_from, ctl_stream_t stream) {
  CTL_CHECK_ARG(x && weight && bias && out, "null pointer");
  CTL_CHECK_ARG(n >= 1 && h >= 1 && w >= 1, "bad activation shape");
  CTL_CHECK_ARG(cin % 64 == 0 && cout % 64 == 0, "Cin=%d and Cout=%d must be multiples of 64", cin, cout);
  CTL_CHECK_ARG(cout <= 2048, "Cout=%d exceeds 2048 (bias staging)", cout);
  CTL_CHECK_ARG((ksize == 1 || ksize == 3) && (stride == 1 || stride == 2), "only 1x1 / 3x3, stride 1 / 2");
  CTL_CHECK_ARG(relu_from % 32 == 0, "relu_from=%d must be a multiple of 32", relu_from);
  int rc = ctl_device_check();
  if (rc) return rc;
  const int pad = ksize == 3 ? 1 : 0;
  const int Ho = (h + 2 * pad - ksize) / stride + 1, Wo = (w + 2 * pad - ksize) / stride + 1;
  {
    static const int c64_mode = [] { const char* e = getenv("CTL_CONV_C64"); return e ? atoi(e) : 1; }();
    if (c64_mode && ksize == 3 && stride == 1 && cin == 64 && cout == 64 && !residual && relu_from == 0)
      return launch_c64(x, n, h, w, weight, bias, out, relu, (cudaStream_t)stream);
  }
  ConvKernelParams p = {};
  pick_tile(Ho, Wo, &p.TH, &p.TW);
  p.tiles_h = (Ho + p.TH - 1) / p.TH;
  p.tiles_w = (Wo + p.TW - 1) / p.TW;
  if ((rc = encode_source(p.a_map, 4, x, n, h, w, cin, stride, p.TH, p.TW))) return rc;
  p.n_taps = 0;
  for (int r = 0; r < ksize; ++r)
    for (int s = 0; s < ksize; ++s) {
      if (stride == 1) {
        p.taps[p.n_taps++] = ConvTap{0, r - pad, s - pad, (r * ksize + s) * cin, cin / 64};
      } else {
        // input row 2*ho + r - pad = 2*(ho + dh) + ph
        const int ar = r - pad, as = s - pad;
        const int ph = ((ar % 2) + 2) % 2, pw = ((as % 2) + 2) % 2;
        const int dh = (ar - ph) / 2, dw = (as - pw) / 2;
        // a tap on an empty parity view reads only padding: it adds exactly zero, so it is not issued
        if (parity_extent(h, ph) == 0 || parity_extent(w, pw) == 0) continue;
        p.taps[p.n_taps++] = ConvTap{ph * 2 + pw, dh, dw, (r * ksize + s) * cin, cin / 64};
      }
    }
  p.k_blocks = p.n_taps * (cin / 64);
  return finish_and_launch(p, n, Ho, Wo, cout, ksize * ksize * cin, weight, bias, residual, out, relu, relu_from,
                           (cudaStream_t)stream);
}

int ctl_conv1x1_dual_nhwc_f16(const void* x1, int32_t cin1, const void* x2, int32_t h2, int32_t w2, int32_t cin2,
                              int32_t stride2, int32_t n, const void* weight_cat, const float* bias, void* out,
                              int32_t cout, int32_t relu, ctl_stream_t stream) {
  CTL_CHECK_ARG(x1 && x2 && weight_cat && bias && out, "null pointer");
  CTL_CHECK_ARG(n >= 1 && h2 >= 1 && w2 >= 1, "bad activation shape");
  CTL_CHECK_ARG(cin1 % 64 == 0 && cin2 % 64 == 0 && cout % 64 == 0 && cin1 >= 64 && cin2 >= 64,
                "Cin1=%d, Cin2=%d and Cout=%d must be multiples of 64", cin1, cin2, cout);
  CTL_CHECK_ARG(cout <= 2048, "Cout=%d exceeds 2048 (bias staging)", cout);
  CTL_CHECK_ARG(stride2 == 1 || (stride2 == 2 && h2 % 2 == 0 && w2 % 2 == 0), "stride2 must be 1, or 2 with even H2, W2");
  int rc = ctl_device_check();
  if (rc) return rc;
  const int Ho = h2 / stride2, Wo = w2 / stride2;
  ConvKernelParams p = {};
  pick_tile(Ho, Wo, &p.TH, &p.TW);
  p.tiles_h = (Ho + p.TH - 1) / p.TH;
  p.tiles_w = (Wo + p.TW - 1) / p.TW;
  // map 0: x1 at the output resolution; map 1: x2 (its (0, 0) parity view when strided); maps 2, 3 unused
  if ((rc = encode_source(&p.a_map[0], 1, x1, n, Ho, Wo, cin1, 1, p.TH, p.TW))) return rc;
  if ((rc = encode_source(&p.a_map[1], 1, x2, n, h2, w2, cin2, stride2, p.TH, p.TW))) return rc;
  p.a_map[2] = p.a_map[0];
  p.a_map[3] = p.a_map[0];
  p.n_taps = 2;
  p.taps[0] = ConvTap{0, 0, 0, 0, cin1 / 64};
  p.taps[1] = ConvTap{1, 0, 0, cin1, cin2 / 64};
  p.k_blocks = (cin1 + cin2) / 64;
  return finish_and_launch(p, n, Ho, Wo, cout, cin1 + cin2, weight_cat, bias, nullptr, out, relu, 0, (cudaStream_t)stream);
}

int ctl_stem_conv7x7(const float* x_nchw, int32_t n, int32_t h, int32_t w, const float* weight_k64, const float* bias,
                     int32_t relu, void* out_nhwc_f16, ctl_stream_t stream) {
  CTL_CHECK_ARG(x_nchw && weight_k64 && bias && out_nhwc_f16, "null pointer");
  CTL_CHECK_ARG(n >= 1 && h >= 7 && w >= 7, "bad input shape");
  int rc = ctl_device_check();
  if (rc) return rc;
  const int Ho = (h + 6 - 7) / 2 + 1, Wo = (w + 6 - 7) / 2 + 1;
  static bool attr_set = false;
  if (!attr_set) {
    CTL_CUDA(cudaFuncSetAttribute(stem_conv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STEM_SMEM));
    attr_set = true;
  }
  dim3 grid((Wo + ST_TW - 1) / ST_TW, (Ho + ST_TH - 1) / ST_TH, n);
  stem_conv_kernel<<<grid, 256, STEM_SMEM, (cudaStream_t)stream>>>(x_nchw, h, w, weight_k64, bias, relu,
                                                                  static_cast<__half*>(out_nhwc_f16), Ho, Wo);
  CTL_LAUNCH_CHECK();
  return 0;
}

int ctl_stem_conv7x7_tc(const float* x_nchw, int32_t n, int32_t h, int32_t w, const void* weight_k192_f16,
                        const float* bias, int32_t relu, void* out_nhwc_f16, ctl_stream_t stream) {
  CTL_CHECK_ARG(x_nchw && weight_k192_f16 && bias && out_nhwc_f16, "null pointer");
  CTL_CHECK_ARG(n >= 1 && h >= 7 && w >= 7, "bad input shape");
  int rc = ctl_device_check();
  if (rc) return rc;
  StemParams p = {};
  p.x = x_nchw;
  p.bias = bias;
  p.out = static_cast<__half*>(out_nhwc_f16);
  p.n_img = n;
  p.H = h;
  p.W = w;
  p.Ho = (h + 6 - 7) / 2 + 1;
  p.Wo = (w + 6 - 7) / 2 + 1;
  p.tiles_h = (p.Ho + S_TH - 1) / S_TH;
  p.tiles_w = (p.Wo + S_TW - 1) / S_TW;
  p.relu = relu;
  const uint64_t dims[2] = {SK, 64};
  const uint64_t strd[2] = {2, SK * 2};
  const uint32_t box[2] = {64, 64};
  if ((rc = encode_tensor_map(&p.w_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 2, weight_k192_f16, dims, strd, box,
                              CU_TENSOR_MAP_SWIZZLE_128B)))
    return rc;
  {
    const uint64_t odims[4] = {64, (uint64_t)p.Wo, (uint64_t)p.Ho, (uint64_t)n};
    const uint64_t ostr[4] = {2, 128, (uint64_t)p.Wo * 128, (uint64_t)p.Ho * p.Wo * 128};
    const uint32_t obox[4] = {64, S_TW, S_TH, 1};
    if ((rc = encode_tensor_map(&p.out_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 4, out_nhwc_f16, odims, ostr, obox,
                                CU_TENSOR_MAP_SWIZZLE_128B)))
      return rc;
  }
  static bool attr_set = false;
  if (!attr_set) {
    CTL_CUDA(cudaFuncSetAttribute(stem_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STEM_TC_SMEM));
    attr_set = true;
  }
  const long long tiles = (long long)n * p.tiles_h * p.tiles_w;
  const int grid = (int)std::min<long long>(tiles, (long long)sm_count());
  CTL_CUDA(launch_k(stem_tc_kernel, dim3(grid), dim3(STEM_TC_THREADS), STEM_TC_SMEM, (cudaStream_t)stream, p));
  CTL_LAUNCH_CHECK();
  return 0;
}

size_t ctl_stem_pad_bytes(int32_t n, int32_t h, int32_t w) {
  (void)w;
  if (n < 1 || h < 1) return 0;
  return (size_t)n * (h + 6) * S3_WP * 4 * sizeof(__half) + 256;  // + slack: the last piece of a row is read 256 B wide
}

// the conv + pool kernel on an already packed input (shared by the fp32 and the uint8 entry points)
static int stem_pool_launch(int32_t n, int32_t h, int32_t w, void* xpad, const void* weight_packed_f16, const float* bias,
                            int32_t relu, void* out_pooled_nhwc_f16, cudaStream_t st) {
  int rc;
  Stem3Params p = {};
  p.w = static_cast<const __half*>(weight_packed_f16);
  p.bias = bias;
  p.out = static_cast<__half*>(out_pooled_nhwc_f16);
  p.n_img = n;
  const int Ho = h / 2;
  p.Wo = w / 2;
  p.hp = Ho / 2;
  p.wp = (p.Wo + 2 - 3) / 2 + 1;
  p.relu = relu;
  const uint64_t pitch = (uint64_t)S3_WP * 8, hp_rows = (uint64_t)h + 6;
  // overlapping view: piece g of a row starts 128 bytes (16 pixels) after piece g-1 and is 192 bytes long
  const uint64_t dims[5] = {(uint64_t)S3_WP * 4, 8, hp_rows / 2, 2, (uint64_t)n};
  const uint64_t strd[5] = {2, 128, 2 * pitch, pitch, hp_rows * pitch};
  const uint32_t box[5] = {S3_PIECE / 2, 8, 5, 1, 1};
  if ((rc = encode_tensor_map(&p.x_map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, 5, xpad, dims, strd, box, CU_TENSOR_MAP_SWIZZLE_NONE)))
    return rc;
  static bool attr_set = false;
  if (!attr_set) {
    CTL_CUDA(cudaFuncSetAttribute(stem_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S3_SMEM));
    attr_set = true;
  }
  const long long tiles = (long long)n * p.hp;
  const int grid = (int)std::min<long long>(tiles, (long long)sm_count());
  CTL_CUDA(launch_k(stem_pool_kernel, dim3(grid), dim3(S3_THREADS), S3_SMEM, st, p));
  return 0;
}

static int stem_fused_check(const void* x, int32_t n, int32_t h, int32_t w, const void* xpad, const void* wt, const float* bias,
                            const void* out) {
  CTL_CHECK_ARG(x && xpad && wt && bias && out, "null pointer");
  CTL_CHECK_ARG(n >= 1 && h >= 8 && w >= 8 && h % 4 == 0 && w % 2 == 0 && w <= 128,
                "the fused stem needs h % 4 == 0, even w <= 128 (use ctl_stem_conv7x7_tc + ctl_maxpool3x3s2_nhwc_f16)");
  return ctl_device_check();
}

int ctl_stem_pool_fused(const float* x_nchw, int32_t n, int32_t h, int32_t w, void* xpad, const void* weight_packed_f16,
                        const float* bias, int32_t relu, void* out_pooled_nhwc_f16, ctl_stream_t stream) {
  int rc = stem_fused_check(x_nchw, n, h, w, xpad, weight_packed_f16, bias, out_pooled_nhwc_f16);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CTL_CUDA(launch_k(stem_pack_input_kernel, dim3((unsigned)(((size_t)n * h + 3) / 4)), dim3(256), 0, st, x_nchw, (int)n, (int)h,
                    (int)w, static_cast<__half*>(xpad)));
  return stem_pool_launch(n, h, w, xpad, weight_packed_f16, bias, relu, out_pooled_nhwc_f16, st);
}

int ctl_stem_pool_fused_u8(const void* x_u8_nhwc, int32_t n, int32_t h, int32_t w, const float* mean3_host, const float* std3_host,
                           void* xpad, const void* weight_packed_f16, const float* bias, int32_t relu, void* out_pooled_nhwc_f16,
                           ctl_stream_t stream) {
  CTL_CHECK_ARG(mean3_host && std3_host, "null pointer");
  CTL_CHECK_ARG(std3_host[0] > 0 && std3_host[1] > 0 && std3_host[2] > 0, "std must be positive");
  int rc = stem_fused_check(x_u8_nhwc, n, h, w, xpad, weight_packed_f16, bias, out_pooled_nhwc_f16);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CTL_CUDA(launch_k(stem_pack_input_u8_kernel, dim3((unsigned)(((size_t)n * h + 3) / 4)), dim3(256), 0, st,
                    static_cast<const uint8_t*>(x_u8_nhwc), (int)n, (int)h, (int)w, mean3_host[0], mean3_host[1], mean3_host[2],
                    std3_host[0], std3_host[1], std3_host[2], static_cast<__half*>(xpad)));
  return stem_pool_launch(n, h, w, xpad, weight_packed_f16, bias, relu, out_pooled_nhwc_f16, st);
}

int ctl_maxpool3x3s2_nhwc_f16(const void* x, int32_t n, int32_t h, int32_t w, int32_t c, void* out,
                              ctl_stream_t stream) {
  CTL_CHECK_ARG(x && out && c % 8 == 0, "bad arguments");
  int rc = ctl_device_check();
  if (rc) return rc;
  const int Ho = (h + 2 - 3) / 2 + 1, Wo = (w + 2 - 3) / 2 + 1;
  const size_t total = (size_t)n * Ho * Wo * (c / 8);
  CTL_CUDA(launch_k(maxpool3x3s2_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, (cudaStream_t)stream,
                    static_cast<const __half*>(x), (int)n, (int)h, (int)w, (int)c, static_cast<__half*>(out), Ho, Wo));
  CTL_LAUNCH_CHECK();
  return 0;
}

int ctl_gap_bn_nhwc_f16(const void* x, int32_t n, int32_t hw, int32_t c, const float* bn_scale, const float* bn_shift,
                        float* feat, float* emb, ctl_stream_t stream) {
  CTL_CHECK_ARG(x && (feat || emb) && c % 2 == 0, "bad arguments");
  CTL_CHECK_ARG(emb == nullptr || (bn_scale && bn_shift), "emb needs the folded BatchNorm1d scale/shift");
  int rc = ctl_device_check();
  if (rc) return rc;
  dim3 grid((c / 2 + 255) / 256, n);
  CTL_CUDA(launch_k(gap_bn_kernel, grid, dim3(256), 0, (cudaStream_t)stream, static_cast<const __half*>(x), (int)hw, (int)c,
                    bn_scale, bn_shift, feat, emb));
  CTL_LAUNCH_CHECK();
  return 0;
}

int ctl_instnorm_relu_nhwc_f16(void* x, int32_t n, int32_t hw, int32_t c, int32_t half, const float* gamma,
                               const float* beta, float eps, ctl_stream_t stream) {
  CTL_CHECK_ARG(x && gamma && beta && half % 8 == 0 && half <= c && c % 8 == 0, "bad arguments");
  int rc = ctl_device_check();
  if (rc) return rc;
  dim3 grid(half / 8, n);
  CTL_CUDA(launch_k(instnorm_relu_kernel, grid, dim3(256), 0, (cudaStream_t)stream, static_cast<__half*>(x), (int)hw, (int)c,
                    (int)half, gamma, beta, eps));
  CTL_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
