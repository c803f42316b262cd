// Shared pieces of the tcgen05 implicit-GEMM convolution kernels (conv3x3_halo.cu, conv_stage1_fused.cu,
// conv_first_tc.cu): tile geometry, parameters, tile decode and the epilogue (TMEM -> registers -> bias / ReLU / mask /
// split-bf16 / projections -> global).
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace osvos {

constexpr int kTileW = 8;     // pixels per patch row  (= one 8-row swizzle atom)
constexpr int kTileH = 16;    // patch rows
constexpr int kBlockM = 128;  // kTileW * kTileH
constexpr int kBlockK = 64;   // channels per K block (128 B of bf16)
constexpr int kABytes = kBlockM * kBlockK * 2;  // 16 KiB per plane

struct ConvParams {
  const float* bias;
  __nv_bfloat16* y_hi;
  __nv_bfloat16* y_lo;
  float* y_f32;
  const __nv_bfloat16* mask_hi;
  const float* proj_w;
  const float* proj_b;
  float* pq;
  __nv_bfloat16* pool_hi;  // optional fused 2x2 ceil-mode max pool of the output
  __nv_bfloat16* pool_lo;
  float* colsum;           // optional fused per-channel sum of the output (bias gradient), atomically accumulated
  int n, h, w, cin, cout;
  int tiles_x, tiles_y, n_blocks, total_tiles, k_chunks;
  int k_steps;  // tcgen05.mma K steps (of 16 channels) issued per 64-channel chunk: 4, or fewer (k_valid)
  int flags;
  // Timing ablations (OSVOS_ABLATE bit mask, diagnosis only - results are garbage): 1 = no weight TMA loads,
  // 2 = no activation TMA loads, 4 = no tcgen05.mma, 8 = no global stores in the epilogue.  0 in production.
  int ablate;
};

__device__ __forceinline__ void decode_tile(const ConvParams& p, int tile, int& nb, int& tx, int& ty, int& img) {
  nb = tile % p.n_blocks;
  int m = tile / p.n_blocks;
  tx = m % p.tiles_x;
  m /= p.tiles_x;
  ty = m % p.tiles_y;
  img = m / p.tiles_y;
}

// Epilogue of one warp (TMEM lane quarter q = warp & 3) over all tiles of this CTA.
__device__ __forceinline__ uint32_t sw128_offset(int row, int chunk) { return row * 128 + ((chunk ^ (row & 7)) << 4); }
__device__ __forceinline__ void epilogue_bar_sync(int nthreads) {
  asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

// Two floats -> packed bf16x2 "hi" word (one F2FP) and the packed residual "lo" word: v ~= hi + lo.
__device__ __forceinline__ void split_pack2(float a, float b, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));            // upper half <- b, lower half <- a
  const float ra = a - __uint_as_float(hi << 16);
  const float rb = b - __uint_as_float(hi & 0xFFFF0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(rb), "f"(ra));
}

// Number of epilogue warps: 8 (two per TMEM lane quarter, each taking every other 32-column chunk) for
// BLOCK_N >= 64, 4 for the N = 16 side-branch kernel.  The epilogue is instruction-bound (~125 cycles per
// output column per tile with 4 warps), which made it the bottleneck of every small-K layer.
template <int BLOCK_N>
struct EpiCfg {
  static constexpr int kGroups = BLOCK_N >= 64 ? 2 : 1;
  static constexpr int kThreads = 128 * kGroups;
};

// Epilogue of one warp over all tiles of this CTA.  Epilogue warps are warps 2 .. 2 + 4*kGroups - 1; warp w
// reads TMEM lane quarter (w & 3) and the 32-column chunks with index parity (w - 2) >> 2.
// SPLIT_ACC: the accumulator stage holds 2 * BLOCK_N columns - [A.B_hi | A.B_lo] produced by one N-concatenated
// tcgen05.mma - and the result is the sum of the two halves.
// The act / pooled / fp32 outputs and the mask of the BLOCK_N >= 64 path move with 256-bit instructions (one full 32-byte
// sector per lane: half the store instructions of the 16-byte form, +2-3 % on inference and fwd+bwd in the round-2 A/B
// - profiles/r02_ab_matrix.txt); every output plane must be 32-byte aligned (checked by osvos_conv3x3).  The bulk-store
// (TMA) epilogue measured the same +2 % at the price of 32 KiB of staging and was dropped.
// TMA_STORE (conv1_1 only, conv_first_tc.cu): the act output goes through `staging` (2 x 16 KiB, 1 KiB aligned) in the
// SWIZZLE_128B layout and leaves with one bulk tensor store per plane and 64-channel slab (full 128-byte rows, image
// edges clipped by the TMA unit) - that layer does nothing but write 105 MB.
template <int BLOCK_N, bool SPLIT_ACC = false, bool TMA_STORE = false>
__device__ __forceinline__ void conv_epilogue_loop(const ConvParams& p, uint32_t tmem_base, uint64_t* tfull_bar,
                                                   uint64_t* tempty_bar, int warp, int lane,
                                                   const CUtensorMap* map_y_hi = nullptr,
                                                   const CUtensorMap* map_y_lo = nullptr, uint8_t* staging = nullptr) {
  constexpr int kEpiThreads = EpiCfg<BLOCK_N>::kThreads;
  const bool epi_leader = (warp == 2) && (lane == 0);
  const int group = (warp - 2) >> 2;
  const int q = warp & 3;  // TMEM lane quarter this warp may read
  const int row = q * 32 + lane;
  const int ly = row / kTileW, lx = row % kTileW;
  const bool relu = (p.flags & OSVOS_FLAG_RELU) != 0;
  const bool masked = (p.flags & OSVOS_FLAG_RELU_MASK) != 0;
  const bool store_ok = !(p.ablate & 8);
  int it = 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
    int nb, tx, ty, img;
    decode_tile(p, tile, nb, tx, ty, img);
    const int as = it & 1;
    const uint32_t aph = (it >> 1) & 1;
    const int y = ty * kTileH + ly, x = tx * kTileW + lx;
    const bool valid = (y < p.h) && (x < p.w) && store_ok;
    const size_t pix = (static_cast<size_t>(img) * p.h + y) * p.w + x;

    mbar_wait(&tfull_bar[as], aph);
    tc_fence_after();
    constexpr int kAccCols = SPLIT_ACC ? 2 * BLOCK_N : BLOCK_N;
    const uint32_t taddr = tmem_base + as * kAccCols + (static_cast<uint32_t>(q * 32) << 16);
    if constexpr (BLOCK_N == 16) {
      uint32_t v[16];
      tmem_ld16(taddr, v);
      uint32_t v2[16];
      if (SPLIT_ACC) tmem_ld16(taddr + 16, v2);
      tmem_ld_wait();
      if (valid) {
        float f[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          f[j] = __uint_as_float(v[j]) + (SPLIT_ACC ? __uint_as_float(v2[j]) : 0.f) + (p.bias ? __ldg(p.bias + j) : 0.f);
          if (relu) f[j] = fmaxf(f[j], 0.f);
        }
        if (p.y_f32) {
          float4* dst = reinterpret_cast<float4*>(p.y_f32 + pix * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) dst[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
        }
        if (p.y_hi) {
          uint32_t hi[8], lo[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) split_pack2(f[2 * j], f[2 * j + 1], hi[j], lo[j]);
          uint4* dh = reinterpret_cast<uint4*>(p.y_hi + pix * 16);
          dh[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          dh[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
          if (p.y_lo) {
            uint4* dl = reinterpret_cast<uint4*>(p.y_lo + pix * 16);
            dl[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
            dl[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
          }
        }
        if (p.pq) {
          float sp = p.proj_b ? __ldg(p.proj_b) : 0.f, sq = 0.f;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            sp = fmaf(f[j], __ldg(p.proj_w + j), sp);
            sq = fmaf(f[j], __ldg(p.proj_w + 16 + j), sq);
          }
          *reinterpret_cast<float2*>(p.pq + pix * 2) = make_float2(sp, sq);
        }
      }
    } else {
#pragma unroll 1
      for (int slab = 0; slab < BLOCK_N / 64; ++slab) {
        const int c0 = slab * 64 + group * 32;     // this warp's 32-column chunk of the 64-column slab
        const int ch = nb * BLOCK_N + c0;
        uint32_t v[32];
        tmem_ld32(taddr + c0, v);
        uint32_t v2[32];
        if (SPLIT_ACC) tmem_ld32(taddr + BLOCK_N + c0, v2);
        float f[32];
        if (p.bias) {
          const float4* bp = reinterpret_cast<const float4*>(p.bias + ch);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = __ldg(bp + j);
            f[4 * j] = b4.x, f[4 * j + 1] = b4.y, f[4 * j + 2] = b4.z, f[4 * j + 3] = b4.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = 0.f;
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          f[j] += __uint_as_float(v[j]);
          if (SPLIT_ACC) f[j] += __uint_as_float(v2[j]);
          f[j] = relu ? fmaxf(f[j], 0.f) : f[j];
        }
        if (masked && valid) {   // two 32-byte loads of the mask's hi plane
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            uint32_t mw[8];
            ld_global_nc_256(p.mask_hi + pix * p.cout + ch + 16 * j, mw);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              if (!(bf16_lo_to_float(mw[t]) > 0.f)) f[16 * j + 2 * t] = 0.f;
              if (!(bf16_hi_to_float(mw[t]) > 0.f)) f[16 * j + 2 * t + 1] = 0.f;
            }
          }
        }
        if (p.y_f32 && valid) {
          float* dst = p.y_f32 + pix * p.cout + ch;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            st_global_256(dst + 8 * j, __float_as_uint(f[8 * j]), __float_as_uint(f[8 * j + 1]), __float_as_uint(f[8 * j + 2]),
                          __float_as_uint(f[8 * j + 3]), __float_as_uint(f[8 * j + 4]), __float_as_uint(f[8 * j + 5]),
                          __float_as_uint(f[8 * j + 6]), __float_as_uint(f[8 * j + 7]));
        }
        if (p.y_hi) {
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) split_pack2(f[2 * j], f[2 * j + 1], hi[j], lo[j]);
          if constexpr (TMA_STORE) {
            // the previous slab's bulk store must have finished READING the staging buffer
            if (epi_leader) tma_store_wait_read<0>();
            epilogue_bar_sync(kEpiThreads);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t off = sw128_offset(row, group * 4 + j);
              *reinterpret_cast<uint4*>(staging + off) = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
              if (p.y_lo)
                *reinterpret_cast<uint4*>(staging + kABytes + off) =
                    make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
            }
            fence_proxy_async_smem();
            epilogue_bar_sync(kEpiThreads);
            if (epi_leader) {
              const int c64 = nb * BLOCK_N + slab * 64;
              tma_store_4d(map_y_hi, staging, c64, tx * kTileW, ty * kTileH, img);
              if (p.y_lo) tma_store_4d(map_y_lo, staging + kABytes, c64, tx * kTileW, ty * kTileH, img);
              tma_store_commit();
            }
          } else if (valid) {
            __nv_bfloat16* dh = p.y_hi + pix * p.cout + ch;
#pragma unroll
            for (int j = 0; j < 2; ++j)
              st_global_256(dh + 16 * j, hi[8 * j], hi[8 * j + 1], hi[8 * j + 2], hi[8 * j + 3], hi[8 * j + 4], hi[8 * j + 5],
                            hi[8 * j + 6], hi[8 * j + 7]);
            if (p.y_lo) {
              __nv_bfloat16* dl = p.y_lo + pix * p.cout + ch;
#pragma unroll
              for (int j = 0; j < 2; ++j)
                st_global_256(dl + 16 * j, lo[8 * j], lo[8 * j + 1], lo[8 * j + 2], lo[8 * j + 3], lo[8 * j + 4], lo[8 * j + 5],
                              lo[8 * j + 6], lo[8 * j + 7]);
            }
          }
        }
        if (p.colsum) {
          // fused bias gradient: per-channel sum over this warp's 32 pixels as a TRANSPOSING reduction - at every
          // halving step a lane keeps the half of its columns selected by one bit of its lane index and hands the other
          // half to its partner: 16 + 8 + 4 + 2 + 1 = 31 shuffles, after which lane l holds the total of column l
          // (the butterfly-per-column form it replaces took 160), then one atomic per lane
          float cs[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) cs[j] = valid ? f[j] : 0.f;
#pragma unroll
          for (int half = 16; half >= 1; half >>= 1) {
            const bool up = (lane & half) != 0;
#pragma unroll
            for (int i = 0; i < half; ++i) {
              const float send = up ? cs[i] : cs[half + i];
              const float keep = up ? cs[half + i] : cs[i];
              cs[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
            }
          }
          atomicAdd(p.colsum + ch + lane, cs[0]);
        }
        if (p.pool_hi) {
          // fused MaxPool2d(2, 2, ceil_mode=True): the 2x2 partners are lanes ^1 (x) and ^8 (y) of this warp;
          // out-of-image partners are excluded (ceil mode clips the window).
          const int oh = (p.h + 1) >> 1, ow = (p.w + 1) >> 1;
          const bool writer = valid && !(lx & 1) && !(ly & 1);
          const size_t opix = (static_cast<size_t>(img) * oh + (y >> 1)) * ow + (x >> 1);
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float m0 = valid ? f[2 * j] : -INFINITY, m1 = valid ? f[2 * j + 1] : -INFINITY;
            m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
            m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
            m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 8));
            m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 8));
            split_pack2(m0, m1, hi[j], lo[j]);
          }
          if (writer) {
            __nv_bfloat16* dh = p.pool_hi + opix * p.cout + ch;
#pragma unroll
            for (int j = 0; j < 2; ++j)
              st_global_256(dh + 16 * j, hi[8 * j], hi[8 * j + 1], hi[8 * j + 2], hi[8 * j + 3], hi[8 * j + 4], hi[8 * j + 5],
                            hi[8 * j + 6], hi[8 * j + 7]);
            if (p.pool_lo) {
              __nv_bfloat16* dl = p.pool_lo + opix * p.cout + ch;
#pragma unroll
              for (int j = 0; j < 2; ++j)
                st_global_256(dl + 16 * j, lo[8 * j], lo[8 * j + 1], lo[8 * j + 2], lo[8 * j + 3], lo[8 * j + 4], lo[8 * j + 5],
                              lo[8 * j + 6], lo[8 * j + 7]);
            }
          }
        }
      }
    }
    tc_fence_before();
    mbar_arrive(&tempty_bar[as]);
  }
  if (TMA_STORE && epi_leader) tma_store_wait_all<0>();
}

// LEAN epilogue - the default for plain forward launches (measured +2.9 % on the 480p frame against the general epilogue
// with 16-byte stores, profiles/r02_ab_matrix.txt; OSVOS_HALO_LEAN=0 selects the general epilogue for A/B runs):
// the inference / plain-forward feature set only - bias, ReLU, split-bf16 act output and / or fused 2x2 max pool, exact
// mode with the N-concatenated accumulator - written against what ncu showed of the general epilogue on the Cin <= 128
// layers (profiles/r01f_ncu_stall_by_role.txt):
//  * stores are 256-bit (one full sector per lane and instruction; the 16-byte ones left write-after-read waits on
//    queued STG as the top stall);
//  * the tcgen05.ld of the NEXT 32-column chunk is issued as soon as the current chunk has been folded into f[], so its
//    latency overlaps the split / store / pool work (21 % of the busy samples were waits on the first use);
//  * the accumulator stage is handed back to the MMA warp right after the LAST tcgen05.ld of the tile has landed,
//    before the stores - not at the end of the tile;
//  * no mask / column-sum / fp32 / bulk-store code: ~1/3 of the instruction footprint next to the issuer.
struct NoTileHook {
  __device__ __forceinline__ void operator()(int) const {}
};
// `pre_tile(tile)` runs at the top of every tile iteration, BEFORE the wait for that tile's accumulator: the fused
// stage-1 kernel uses the epilogue warps' idle time there to build conv1_1's operand rows of a later tile.
template <int BLOCK_N, class TileHook = NoTileHook>
__device__ __forceinline__ void conv_epilogue_lean(const ConvParams& p, uint32_t tmem_base, uint64_t* tfull_bar,
                                                   uint64_t* tempty_bar, int warp, int lane, TileHook pre_tile = TileHook()) {
  static_assert(BLOCK_N == 64 || BLOCK_N == 128, "lean epilogue: 64- or 128-wide exact tiles");
  constexpr int kAccCols = 2 * BLOCK_N, kSlabs = BLOCK_N / 64;
  const int group = (warp - 2) >> 2;
  const int q = warp & 3;
  const int row = q * 32 + lane;
  const int ly = row / kTileW, lx = row % kTileW;
  const bool relu = (p.flags & OSVOS_FLAG_RELU) != 0;
  const int oh = (p.h + 1) >> 1, ow = (p.w + 1) >> 1;
  int it = 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
    int nb, tx, ty, img;
    decode_tile(p, tile, nb, tx, ty, img);
    const int as = it & 1;
    const uint32_t aph = (it >> 1) & 1;
    const int y = ty * kTileH + ly, x = tx * kTileW + lx;
    const bool valid = (y < p.h) && (x < p.w);
    const size_t pix = (static_cast<size_t>(img) * p.h + y) * p.w + x;
    const size_t opix = (static_cast<size_t>(img) * oh + (y >> 1)) * ow + (x >> 1);
    const bool writer = valid && !(lx & 1) && !(ly & 1);

    pre_tile(tile);
    mbar_wait(&tfull_bar[as], aph);
    tc_fence_after();
    const uint32_t taddr = tmem_base + as * kAccCols + (static_cast<uint32_t>(q * 32) << 16) + group * 32;
    uint32_t v[32], v2[32];
    tmem_ld32(taddr, v);
    tmem_ld32(taddr + BLOCK_N, v2);
#pragma unroll 1                        // (rolled: the body is ~900 instructions and shares the I-cache with the issuer)
    for (int slab = 0; slab < kSlabs; ++slab) {
      const int ch = nb * BLOCK_N + slab * 64 + group * 32;
      float f[32];
      if (p.bias) {
        const float4* bp = reinterpret_cast<const float4*>(p.bias + ch);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 b4 = __ldg(bp + j);
          f[4 * j] = b4.x, f[4 * j + 1] = b4.y, f[4 * j + 2] = b4.z, f[4 * j + 3] = b4.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = 0.f;
      }
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        f[j] += __uint_as_float(v[j]);        // same association as conv_epilogue_loop: bit-identical outputs
        f[j] += __uint_as_float(v2[j]);
        f[j] = relu ? fmaxf(f[j], 0.f) : f[j];
      }
      if (slab + 1 < kSlabs) {          // next chunk's accumulator columns: in flight behind the work below
        tmem_ld32(taddr + (slab + 1) * 64, v);
        tmem_ld32(taddr + BLOCK_N + (slab + 1) * 64, v2);
      } else {                          // every column of this stage has been read: the MMA warp may reuse it
        tc_fence_before();
        mbar_arrive(&tempty_bar[as]);
      }
      if (p.y_hi) {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) split_pack2(f[2 * j], f[2 * j + 1], hi[j], lo[j]);
        if (valid) {
          __nv_bfloat16* dh = p.y_hi + pix * p.cout + ch;
#pragma unroll
          for (int j = 0; j < 2; ++j)
            st_global_256(dh + 16 * j, hi[8 * j], hi[8 * j + 1], hi[8 * j + 2], hi[8 * j + 3], hi[8 * j + 4], hi[8 * j + 5],
                          hi[8 * j + 6], hi[8 * j + 7]);
          if (p.y_lo) {
            __nv_bfloat16* dl = p.y_lo + pix * p.cout + ch;
#pragma unroll
            for (int j = 0; j < 2; ++j)
              st_global_256(dl + 16 * j, lo[8 * j], lo[8 * j + 1], lo[8 * j + 2], lo[8 * j + 3], lo[8 * j + 4], lo[8 * j + 5],
                            lo[8 * j + 6], lo[8 * j + 7]);
          }
        }
      }
      if (p.pool_hi) {
        // fused MaxPool2d(2, 2, ceil_mode=True): partners are lanes ^1 (x) and ^8 (y); out-of-image partners excluded
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float m0 = valid ? f[2 * j] : -INFINITY, m1 = valid ? f[2 * j + 1] : -INFINITY;
          m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
          m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
          m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 8));
          m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 8));
          split_pack2(m0, m1, hi[j], lo[j]);
        }
        if (writer) {
          __nv_bfloat16* dh = p.pool_hi + opix * p.cout + ch;
#pragma unroll
          for (int j = 0; j < 2; ++j)
            st_global_256(dh + 16 * j, hi[8 * j], hi[8 * j + 1], hi[8 * j + 2], hi[8 * j + 3], hi[8 * j + 4], hi[8 * j + 5],
                          hi[8 * j + 6], hi[8 * j + 7]);
          if (p.pool_lo) {
            __nv_bfloat16* dl = p.pool_lo + opix * p.cout + ch;
#pragma unroll
            for (int j = 0; j < 2; ++j)
              st_global_256(dl + 16 * j, lo[8 * j], lo[8 * j + 1], lo[8 * j + 2], lo[8 * j + 3], lo[8 * j + 4], lo[8 * j + 5],
                            lo[8 * j + 6], lo[8 * j + 7]);
          }
        }
      }
    }
  }
}

// ---- host helpers shared by the launchers ------------------------------------------------
static inline void fill_conv_params(ConvParams& p, const osvos_conv3x3_args* a, int block_n) {
  p.bias = a->bias;
  p.y_hi = static_cast<__nv_bfloat16*>(a->y_hi);
  p.y_lo = static_cast<__nv_bfloat16*>(a->y_lo);
  p.y_f32 = a->y_f32;
  p.mask_hi = static_cast<const __nv_bfloat16*>(a->mask_hi);
  p.proj_w = a->proj_w;
  p.proj_b = a->proj_b;
  p.pq = a->pq;
  p.pool_hi = static_cast<__nv_bfloat16*>(a->pool_hi);
  p.pool_lo = static_cast<__nv_bfloat16*>(a->pool_lo);
  p.colsum = a->colsum;
  p.n = a->n;
  p.h = a->h;
  p.w = a->w;
  p.cin = a->cin;
  p.cout = a->cout;
  p.tiles_x = (a->w + kTileW - 1) / kTileW;
  p.tiles_y = (a->h + kTileH - 1) / kTileH;
  p.n_blocks = a->cout / block_n;
  p.total_tiles = p.tiles_x * p.tiles_y * a->n * p.n_blocks;
  p.k_chunks = a->cin / kBlockK;
  p.k_steps = (a->k_valid > 0 && a->k_valid < kBlockK) ? (a->k_valid + 15) / 16 : kBlockK / 16;
  p.flags = a->flags;
  p.ablate = env_int("OSVOS_ABLATE", 0);
}

int conv_first_tc_launch(const float* x, const float* w_oihw, const float* bias, void* y_hi, void* y_lo, int n, int h,
                         int w, int flags, cudaStream_t stream);
int side_conv_dispatch(const osvos_conv3x3_args* a, cudaStream_t stream);
int side_conv_multi_dispatch(const osvos_conv3x3_args* const* args, int count, cudaStream_t stream);
int conv3x3_halo_dispatch(const osvos_conv3x3_args* a, cudaStream_t stream);

}  // namespace osvos
