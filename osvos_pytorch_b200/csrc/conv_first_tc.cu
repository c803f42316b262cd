// conv1_1 (3 -> 64 channels, 3x3, pad 1) + bias + ReLU on the tensor cores.
//
// K = 27 is too small for TMA-fed operands (and the frame is NCHW fp32), so the im2col A tile is BUILT in
// shared memory by four producer warps straight from the caller's frame: row m = pixel, k = ci*9 + 3r + s,
// split into bf16 hi / lo, written in the canonical K-major SWIZZLE_128B layout (16-byte chunk j of row m
// lands at chunk j ^ (m & 7)).  Only k < 32 is ever written or read: two UMMA K-steps x three passes = 6
// tcgen05.mma per 128-pixel tile.  The 64 x 27 weight matrix is converted once per CTA into the same
// layout (B operand, resident).  Epilogue = the shared conv epilogue (bias, ReLU, split-bf16 act store).
// Generic-proxy smem writes are made visible to the tensor core with fence.proxy.async before the
// mbarrier arrive.
//
// Measured alternatives (round 1): staging the 3 x 18 x 10 input patch in shared memory and gathering the taps from
// it was slower (110 vs 74 us); direct 16-byte global stores instead of the TMA-store epilogue were slower (93 us).
//
// Replaces stages[0][0..1] of the reference (networks/vgg_osvos.py:61,142-143).
#include <string.h>

#include "conv_common.cuh"

namespace osvos {

constexpr int kFirstTcThreads = 448;  // warp 0 idle, warp 1 MMA, warps 2-9 epilogue, warps 10-13 A builders
constexpr int kFirstStages = 3;
constexpr int kFirstStageBytes = 2 * kABytes;           // hi + lo planes of the A tile (128 rows x 128 B each)
constexpr int kFirstBBytes = 2 * 64 * 128;              // hi + lo planes of the weights (64 rows x 128 B)
constexpr int kFirstStagingBytes = 2 * kABytes;         // TMA-store staging (hi + lo slab of the output tile)
constexpr int kFirstSmem = kFirstStages * kFirstStageBytes + kFirstBBytes + kFirstStagingBytes + 1024 + 256;

template <int PLANES>
__global__ void __launch_bounds__(kFirstTcThreads, 1)
conv_first_tc_kernel(const float* __restrict__ x, const float* __restrict__ wgt,
                     const __grid_constant__ CUtensorMap map_y_hi, const __grid_constant__ CUtensorMap map_y_lo,
                     const ConvParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_b = smem + kFirstStages * kFirstStageBytes;
  uint8_t* staging = smem_b + kFirstBBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + kFirstStagingBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kFirstStages;
  uint64_t* tfull_bar = bars + 2 * kFirstStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kFirstStages; ++i) {
      mbar_init(&full_bar[i], 128);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], EpiCfg<64>::kThreads);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  // PDL: the weights may have been rewritten by the previous kernel of the stream (the optimizer step), so even
  // the resident B operand is built after the wait; only barrier init and the TMEM allocation overlap its tail.
  pdl_wait();
  pdl_launch_dependents();
  // resident B operand: rows = co, k = ci*9 + 3r + s (the OIHW flattening), chunks 0..3 (k < 32)
  for (int i = threadIdx.x; i < 64 * 4; i += kFirstTcThreads) {
    const int co = i >> 2, chunk = i & 3;
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int k0 = chunk * 8 + 2 * t;
      const float v0 = k0 < 27 ? wgt[co * 27 + k0] : 0.f;
      const float v1 = k0 + 1 < 27 ? wgt[co * 27 + k0 + 1] : 0.f;
      __nv_bfloat16 h0, l0, h1, l1;
      split_bf16(v0, h0, l0);
      split_bf16(v1, h1, l1);
      hi[t] = pack_bf16x2(h0, h1);
      lo[t] = pack_bf16x2(l0, l1);
    }
    *reinterpret_cast<uint4*>(smem_b + sw128_offset(co, chunk)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(smem_b + 64 * 128 + sw128_offset(co, chunk)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 1) {
    // -------------------------------------------------------------- MMA issuer (one elected thread, see conv3x3_halo.cu)
    if (elect_one()) {
    constexpr uint32_t idesc = make_idesc_f16(kBlockM, 64, /*bf16=*/true);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      mbar_wait(&tempty_bar[as], aph ^ 1);
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      {
        const uint32_t tmem_d = tmem_base + as * 64;
        const uint32_t a_hi = smem_u32(smem + stage * kFirstStageBytes);
        const uint32_t b_hi = smem_u32(smem_b);
        const uint64_t da_hi = make_smem_desc(a_hi, 16, 1024, kLayoutSW128);
        const uint64_t da_lo = make_smem_desc(a_hi + kABytes, 16, 1024, kLayoutSW128);
        const uint64_t db_hi = make_smem_desc(b_hi, 16, 1024, kLayoutSW128);
        const uint64_t db_lo = make_smem_desc(b_hi + 64 * 128, 16, 1024, kLayoutSW128);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const uint64_t adv = static_cast<uint64_t>(k * 2);
          if (PLANES == 2) {
            umma_f16(tmem_d, da_lo + adv, db_hi + adv, idesc, k != 0);
            umma_f16(tmem_d, da_hi + adv, db_lo + adv, idesc, 1);
            umma_f16(tmem_d, da_hi + adv, db_hi + adv, idesc, 1);
          } else {
            umma_f16(tmem_d, da_hi + adv, db_hi + adv, idesc, k != 0);
          }
        }
        umma_commit(&empty_bar[stage]);
        umma_commit(&tfull_bar[as]);
      }
      if (++stage == kFirstStages) {
        stage = 0;
        phase ^= 1;
      }
    }
    }
    __syncwarp();
  } else if (warp >= 2 && warp < 10) {
    conv_epilogue_loop<64, false, true>(p, tmem_base, tfull_bar, tempty_bar, warp, lane, &map_y_hi, &map_y_lo, staging);
  } else if (warp >= 10) {
    // ------------------------------------------------------------- A builders
    const int row = (warp - 10) * 32 + lane;  // GEMM row = pixel of the tile
    const int ly = row / kTileW, lx = row % kTileW;
    int stage = 0;
    uint32_t phase = 0;
    const size_t plane_sz = static_cast<size_t>(p.h) * p.w;
    // Register double buffering: the 27 taps of the NEXT tile are requested before the current tile is converted and
    // written, so the global-load latency (the builders handle one tile at a time) overlaps the shared-memory work
    // and the wait for a free stage instead of being paid once per tile.
    auto load_tile = [&](int tile, float (&v)[27]) {
      int nb, tx, ty, img;
      decode_tile(p, tile, nb, tx, ty, img);
      const int y = ty * kTileH + ly, xx = tx * kTileW + lx;
#pragma unroll
      for (int ci = 0; ci < 3; ++ci) {
        const float* pl = x + (static_cast<size_t>(img) * 3 + ci) * plane_sz;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const int iy = y + r - 1;
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            const int ix = xx + s - 1;
            v[ci * 9 + r * 3 + s] =
                (iy >= 0 && iy < p.h && ix >= 0 && ix < p.w) ? __ldg(pl + static_cast<size_t>(iy) * p.w + ix) : 0.f;
          }
        }
      }
    };
    float vn[27];
    if (static_cast<int>(blockIdx.x) < p.total_tiles) load_tile(blockIdx.x, vn);
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      float v[32];
#pragma unroll
      for (int k = 0; k < 27; ++k) v[k] = vn[k];
#pragma unroll
      for (int k = 27; k < 32; ++k) v[k] = 0.f;
      if (tile + static_cast<int>(gridDim.x) < p.total_tiles) load_tile(tile + gridDim.x, vn);
      mbar_wait(&empty_bar[stage], phase ^ 1);
      uint8_t* st = smem + stage * kFirstStageBytes;
#pragma unroll
      for (int chunk = 0; chunk < 4; ++chunk) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          __nv_bfloat16 h0, l0, h1, l1;
          split_bf16(v[chunk * 8 + 2 * t], h0, l0);
          split_bf16(v[chunk * 8 + 2 * t + 1], h1, l1);
          hi[t] = pack_bf16x2(h0, h1);
          lo[t] = pack_bf16x2(l0, l1);
        }
        *reinterpret_cast<uint4*>(st + sw128_offset(row, chunk)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        if (PLANES == 2)
          *reinterpret_cast<uint4*>(st + kABytes + sw128_offset(row, chunk)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
      fence_proxy_async_smem();
      mbar_arrive(&full_bar[stage]);
      if (++stage == kFirstStages) {
        stage = 0;
        phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

int conv_first_tc_launch(const float* x, const float* w_oihw, const float* bias, void* y_hi, void* y_lo, int n, int h,
                         int w, int flags, cudaStream_t stream) {
  osvos_conv3x3_args a;
  memset(&a, 0, sizeof(a));
  a.bias = bias;
  a.y_hi = y_hi;
  a.y_lo = (flags & OSVOS_FLAG_FAST) ? nullptr : y_lo;
  a.n = n;
  a.h = h;
  a.w = w;
  a.cin = 64;  // unused by the epilogue; keeps k_chunks well defined
  a.cout = 64;
  a.flags = flags;
  ConvParams p;
  fill_conv_params(p, &a, 64);
  CUtensorMap my_hi, my_lo;   // the act output's bulk-store maps
  const int rc = encode_act_maps(&my_hi, &my_lo, a.y_hi, a.y_lo, n, h, w, 64, kTileW, kTileH);
  if (rc) return rc;
  OSVOS_CHECK_CUDA((flags & OSVOS_FLAG_FAST)
                       ? launch_persistent<conv_first_tc_kernel<1>>(p.total_tiles, kFirstTcThreads, kFirstSmem, stream, x,
                                                                    w_oihw, my_hi, my_lo, p)
                       : launch_persistent<conv_first_tc_kernel<2>>(p.total_tiles, kFirstTcThreads, kFirstSmem, stream, x,
                                                                    w_oihw, my_hi, my_lo, p));
  return OSVOS_OK;
}

}  // namespace osvos
