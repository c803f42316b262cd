// Stage 1 of the trunk as ONE kernel (inference): conv1_1 (3 -> 64, + bias + ReLU) computed INSIDE conv1_2's kernel,
// on the 18 x 10-pixel halo patch conv1_2 reads anyway, so that the 105 MB split-bf16 map between the two layers is
// never written to or read from memory (separately the two kernels took 51 + 82 us of a 790 us frame, conv1_1 being
// nothing but that write).  Replaces stages[0] of the reference (networks/vgg_osvos.py:61,140-143: conv, ReLU, conv,
// ReLU) and the first max pool (:140) when the caller only needs the pooled output.
//
// conv1_2 part = conv3x3_halo_kernel<64, exact, lean epilogue> unchanged: nine taps as nine UMMA descriptors into the
// halo patch, weight slabs streamed by TMA through a ring, N-concatenated split accumulator, lean epilogue with the
// fused 2 x 2 max pool.  What changes is WHO fills the activation stage: not a TMA box but the CTA itself:
//   1. (the eight conv1_2 epilogue warps, in their idle time) build the im2col operand of conv1_1 for the 180 halo pixels (rows m = hy * 10 + hx, k = ci * 9 + 3r + s < 27,
//      split bf16 hi / lo, canonical K-major SWIZZLE_128B rows - the layout of conv_first_tc.cu) from the fp32 frame;
//   2. the MMA warp runs conv1_1 on it: two M = 128 halves x two K steps x (A_hi.[B_hi | B_lo] + A_lo.B_hi) into 2 x 128
//      TMEM columns next to conv1_2's two accumulator stages (512 columns in all);
//      (pixels 128 .. 179 sit at rows 192 .. 243 of the operand, i.e. in TMEM lanes 64 .. 115 of the second M half, so that
//      six warps - lane quarters 2, 3, 0, 1, 2, 3 - own exactly one pixel per thread);
//   3. six "stage-1" warps read those accumulators back, add the bias, apply ReLU, ZERO the halo pixels that lie outside the
//      image (they are conv1_2's zero padding, not conv1_1 evaluated outside the frame), split into hi / lo and write
//      the rows of the activation stage exactly where the TMA box of the unfused kernel would have put them
//      (generic-proxy writes + fence.proxy.async before the mbarrier arrive).
// Issue order per tile j: [conv1_1 MMAs of tile j + 1] then [conv1_2 MMAs of tile j], so that steps 3 and 1 of the
// stage-1 warps hide behind the 4 k cycles of conv1_2's MMAs.  Single-buffered im2col tile and conv1_1 accumulators.
// History (profiles/r02c .. r02h): v1 - four stage-1 warps doing steps 1 and 3 for two pixels each, every load waited
// for in turn: 9 k cycles per tile against 4.5 k of MMAs, no faster than two kernels.  v2 - six warps, one pixel per
// thread, taps of the next tile and the next 16 accumulator columns requested ahead: 7.5 k.  v3 - one base pointer and
// 32-bit offsets for the 27 taps instead of per-tap 64-bit addressing: 6.9 k, the stage-1 warps still the pace of the
// kernel.  v4 (this) - step 1 moved to the epilogue warps, three tiles ahead, so that the stage-1 warps only convert.
#include <string.h>

#include <type_traits>

#include "conv_common.cuh"

namespace osvos {

constexpr int kS1Pitch = 10;                                        // halo patch row pitch in pixels (packed rows)
constexpr int kS1HaloRows = kTileH + 2;                             // 18
constexpr int kS1HaloPx = kS1HaloRows * kS1Pitch;                   // 180 GEMM rows of conv1_1 per tile
constexpr int kS1APlane = (kS1HaloPx * 128 + 1023) / 1024 * 1024;   // 23552 B: one plane of one activation stage
constexpr int kS1AStage = 2 * kS1APlane;
constexpr int kS1AStages = 2;
constexpr int kS1BPlane = 64 * 128;                                 // conv1_2 weight slab, one plane (64 co x 64 ci)
constexpr int kS1BStage = 2 * kS1BPlane;
// The K = 32 operands of conv1_1 (im2col tile, weights) use 64 of the 128 bytes of a SWIZZLE_128B row.  SW64 = true stores
// them as 64-byte rows in the SWIZZLE_64B layout instead (8-row atoms of 512 B, 16-byte chunk c of row r at chunk
// c ^ ((r >> 1) & 3)), which frees 40 KiB for the conv1_2 weight ring: 5 stages instead of 3.  The ring depth is what
// bounds the kernel - a tap's slab is consumed in ~450 cycles but takes ~2000 to arrive from L2, and with two slabs in
// flight the first version ran at 7.2 k cycles per tile against 4.5 k of MMAs (profiles/r02d_*).
template <bool SW64>
struct S1Cfg {
  static constexpr int kRowBytes = SW64 ? 64 : 128;
  static constexpr int kIm2colPlane = 256 * kRowBytes;              // M = 256 rows (k < 32 used)
  static constexpr int kW1Plane = 64 * kRowBytes;
  static constexpr int kW1Bytes = 2 * kW1Plane;                     // conv1_1 weights: [hi 64 rows][lo 64 rows]
  static constexpr int kBStages = SW64 ? 5 : 3;
  static constexpr int kSmem = kS1AStages * kS1AStage + kBStages * kS1BStage + 2 * kIm2colPlane + kW1Bytes + 1024 + 512;
  static constexpr uint64_t kLayout = SW64 ? kLayoutSW64 : kLayoutSW128;
  static constexpr int kSbo = SW64 ? 512 : 1024;                    // bytes between 8-row groups
  static_assert(kSmem <= 227 * 1024, "stage-1 kernel exceeds the per-CTA shared memory");
  static_assert(kSmem + 4096 < (1 << 18), "descriptor start-address field would overflow");
  __device__ static __forceinline__ uint32_t offset(int row, int chunk) {
    return SW64 ? static_cast<uint32_t>(row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4)) : sw128_offset(row, chunk);
  }
};
constexpr int kS1EpiThreads = EpiCfg<64>::kThreads;                 // 256: warps 2 .. 9
constexpr int kS1S1Threads = 192;                                   // stage-1 warps 10 .. 15: one halo pixel per thread
constexpr int kS1Threads = 64 + kS1EpiThreads + kS1S1Threads;

struct Stage1Params {
  const float* x;    // [n,3,h,w] fp32 frame
  const float* w1;   // conv1_1 weight [64,3,3,3]
  const float* b1;   // conv1_1 bias [64] or NULL
};

template <bool SW64>
__global__ void __launch_bounds__(kS1Threads, 1)
conv_stage1_fused_kernel(const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                         const Stage1Params s1, const ConvParams p) {
  using Cfg = S1Cfg<SW64>;
  constexpr int kS1BStages = Cfg::kBStages, kS1Im2colPlane = Cfg::kIm2colPlane;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem_a + kS1AStages * kS1AStage;
  uint8_t* smem_i = smem_b + kS1BStages * kS1BStage;     // im2col operand: [hi plane 256 rows][lo plane 256 rows]
  uint8_t* smem_w1 = smem_i + 2 * kS1Im2colPlane;        // conv1_1 weights [hi 64 rows][lo 64 rows]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_w1 + Cfg::kW1Bytes);
  uint64_t* a_full = bars;                       // [2] stage-1 warps -> MMA   (128 arrivals)
  uint64_t* a_empty = bars + 2;                  // [2] MMA -> stage-1 warps   (commit)
  uint64_t* b_full = bars + 4;                   // [kBStages] TMA -> MMA
  uint64_t* b_empty = bars + 4 + kS1BStages;     // [kBStages] MMA -> TMA producer
  uint64_t* tfull_bar = bars + 4 + 2 * kS1BStages;   // [2] conv1_2 accumulator ready
  uint64_t* tempty_bar = tfull_bar + 2;              // [2] conv1_2 accumulator drained (256 arrivals)
  uint64_t* i_full = tempty_bar + 2;             // im2col tile built              (128 arrivals)
  uint64_t* i_empty = i_full + 1;                // conv1_1 MMAs have read it      (commit)
  uint64_t* c_full = i_empty + 1;                // conv1_1 accumulators ready     (commit)
  uint64_t* c_empty = c_full + 1;                // ... and read back              (128 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(c_empty + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_w_hi);
    tma_prefetch_desc(&map_w_lo);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&a_full[i], kS1S1Threads);
      mbar_init(&a_empty[i], 1);
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], kS1EpiThreads);
    }
    for (int i = 0; i < kS1BStages; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    mbar_init(i_full, kS1EpiThreads);
    mbar_init(i_empty, 1);
    mbar_init(c_full, 1);
    mbar_init(c_empty, kS1S1Threads);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);   // [0,256): two conv1_2 accumulator stages; [256,512): conv1_1, two M halves
  pdl_wait();               // the frame / the weights may come from the previous kernel of the stream
  pdl_launch_dependents();
  // resident B operand of conv1_1: rows = co, k = ci*9 + 3r + s (the OIHW flattening), chunks 0..3 (k < 32)
  for (int i = threadIdx.x; i < 64 * 4; i += kS1Threads) {
    const int co = i >> 2, chunk = i & 3;
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int k0 = chunk * 8 + 2 * t;
      const float v0 = k0 < 27 ? __ldg(s1.w1 + co * 27 + k0) : 0.f;
      const float v1 = k0 + 1 < 27 ? __ldg(s1.w1 + co * 27 + k0 + 1) : 0.f;
      split_pack2(v0, v1, hi[t], lo[t]);
    }
    *reinterpret_cast<uint4*>(smem_w1 + Cfg::offset(co, chunk)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(smem_w1 + Cfg::kW1Plane + Cfg::offset(co, chunk)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_c1 = tmem_base + 256;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer: conv1_2 weight slabs only
    if (elect_one()) {
      int b_stage = 0;
      uint32_t b_phase = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          mbar_wait(&b_empty[b_stage], b_phase ^ 1);
          uint8_t* st = smem_b + b_stage * kS1BStage;
          mbar_arrive_expect_tx(&b_full[b_stage], kS1BStage);
          tma_load_3d(&map_w_hi, &b_full[b_stage], st, 0, 0, tap);
          tma_load_3d(&map_w_lo, &b_full[b_stage], st + kS1BPlane, 0, 0, tap);
          if (++b_stage == kS1BStages) {
            b_stage = 0;
            b_phase ^= 1;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // -------------------------------------------------------------- MMA issuer (one elected thread)
    if (elect_one()) {
      constexpr uint32_t idesc64 = make_idesc_f16(kBlockM, 64, /*bf16=*/true);
      constexpr uint32_t idesc128 = make_idesc_f16(kBlockM, 128, /*bf16=*/true);
      constexpr uint64_t kDescA = (static_cast<uint64_t>(16 >> 4) << 16) | (static_cast<uint64_t>((kS1Pitch * 128) >> 4) << 32) |
                                  (1ull << 46) | (static_cast<uint64_t>(kLayoutSW128) << 61);
      constexpr uint64_t kDescK = (static_cast<uint64_t>(16 >> 4) << 16) | (static_cast<uint64_t>(1024 >> 4) << 32) |
                                  (1ull << 46) | (static_cast<uint64_t>(kLayoutSW128) << 61);   // plain 8-row groups
      // conv1_1's operands: 64- or 128-byte rows (S1Cfg)
      constexpr uint64_t kDescI = (static_cast<uint64_t>(16 >> 4) << 16) | (static_cast<uint64_t>(Cfg::kSbo >> 4) << 32) |
                                  (1ull << 46) | (Cfg::kLayout << 61);
      const uint32_t smem_a_u32 = smem_u32(smem_a), smem_b_u32 = smem_u32(smem_b);
      const uint64_t di_hi = kDescI | static_cast<uint64_t>(smem_u32(smem_i) >> 4);
      const uint64_t di_lo = di_hi + (kS1Im2colPlane >> 4);
      const uint64_t dw1 = kDescI | static_cast<uint64_t>(smem_u32(smem_w1) >> 4);   // [hi | lo]: 128 rows
      uint32_t i_phase = 0, c_phase = 0;
      // conv1_1 of one tile: 2 M halves x 2 K steps x (A_hi.[B_hi | B_lo] (N = 128) + A_lo.B_hi (N = 64))
      auto conv1_1 = [&]() {
        mbar_wait(i_full, i_phase);
        mbar_wait(c_empty, c_phase ^ 1);          // the previous tile's accumulators have been read back
        tc_fence_after();
#pragma unroll
        for (int mh = 0; mh < 2; ++mh) {
          const uint32_t d = tmem_c1 + mh * 128;
          const uint32_t moff = static_cast<uint32_t>(mh * 128 * Cfg::kRowBytes) >> 4;
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            umma_f16(d, di_hi + moff + 2 * k, dw1 + 2 * k, idesc128, k != 0);
            umma_f16(d, di_lo + moff + 2 * k, dw1 + 2 * k, idesc64, 1);
          }
        }
        umma_commit(i_empty);
        umma_commit(c_full);
        i_phase ^= 1;
        c_phase ^= 1;
      };
      int a_stage = 0, b_stage = 0;
      uint32_t a_phase = 0, b_phase = 0;
      int it = 0;
      if (static_cast<int>(blockIdx.x) < p.total_tiles) conv1_1();
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
        if (tile + static_cast<int>(gridDim.x) < p.total_tiles) conv1_1();     // next tile's conv1_1 first
        const int as = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait(&tempty_bar[as], aph ^ 1);
        mbar_wait(&a_full[a_stage], a_phase);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * 128;
        const uint64_t da0 = kDescA | static_cast<uint64_t>((smem_a_u32 + a_stage * kS1AStage) >> 4);
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          const uint32_t tap_off = static_cast<uint32_t>(((tap / 3) * kS1Pitch + (tap % 3)) * (128 >> 4));
          mbar_wait(&b_full[b_stage], b_phase);
          tc_fence_after();
          const uint64_t db_hi = kDescK | static_cast<uint64_t>((smem_b_u32 + b_stage * kS1BStage) >> 4);
          const uint64_t da_hi = da0 + tap_off;
          const uint64_t da_lo = da_hi + (kS1APlane >> 4);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            umma_f16(tmem_d, da_hi + 2 * k, db_hi + 2 * k, idesc128, (tap | k) != 0);   // [A_hi.B_hi | A_hi.B_lo]
            umma_f16(tmem_d, da_lo + 2 * k, db_hi + 2 * k, idesc64, 1);                 // + A_lo.B_hi
          }
          umma_commit(&b_empty[b_stage]);
          if (tap == 8) {
            umma_commit(&a_empty[a_stage]);
            umma_commit(&tfull_bar[as]);
          }
          if (++b_stage == kS1BStages) {
            b_stage = 0;
            b_phase ^= 1;
          }
        }
        if (++a_stage == kS1AStages) {
          a_stage = 0;
          a_phase ^= 1;
        }
      }
    }
    __syncwarp();
  } else if (warp < 2 + kS1EpiThreads / 32) {
    // ------------------------------------------------------------ conv1_2 epilogue (bias, ReLU, act and / or pooled output)
    // ... and, in the time these eight warps otherwise spend waiting for the next accumulator (half of it: profiles/
    // r02a_ncu_stall_by_role_lean.txt), the im2col operand rows of conv1_1: thread t builds the row of halo pixel t
    // (< 180) of the tile THREE tile-steps ahead of the one whose accumulator it is about to read - that tile's conv1_1
    // MMAs are issued one step ahead of its conv1_2 MMAs, which run one step ahead of this epilogue.  The row is built at
    // the top of the iteration (the wait for the previous conv1_1's commit and the latency of the 27 tap loads are paid
    // while the accumulator is still being produced).  One 64-bit base pointer per tile, 32-bit offsets
    // ci * plane + r * w + s, three row and three column predicates (the first version's per-tap 64-bit addressing was
    // 640 of a builder thread's 1200 instructions per tile).
    const int pix = threadIdx.x - 64;                                   // 0 .. 255: halo pixel built by this thread
    const bool live = pix < kS1HaloPx;
    const int irow = pix < 128 ? pix : pix + 64;                        // pixels 128 .. 179 -> operand rows 192 .. 243
    const int hy = pix / kS1Pitch, hx = pix - hy * kS1Pitch;
    const size_t plane_sz = static_cast<size_t>(p.h) * p.w;
    const int fw = p.w, fplane = p.h * p.w;
    uint32_t i_phase = 0;
    int built = 0;                                                      // operand rows built so far (tile ordinal)
    auto build = [&](int tile) {
      int nb, tx, ty, img;
      decode_tile(p, tile, nb, tx, ty, img);
      const int y = ty * kTileH - 1 + hy, xx = tx * kTileW - 1 + hx;
      const bool ry[3] = {live && static_cast<unsigned>(y - 1) < static_cast<unsigned>(p.h),
                          live && static_cast<unsigned>(y) < static_cast<unsigned>(p.h),
                          live && static_cast<unsigned>(y + 1) < static_cast<unsigned>(p.h)};
      const bool cx[3] = {static_cast<unsigned>(xx - 1) < static_cast<unsigned>(fw), static_cast<unsigned>(xx) < static_cast<unsigned>(fw),
                          static_cast<unsigned>(xx + 1) < static_cast<unsigned>(fw)};
      const float* base = s1.x + static_cast<size_t>(img) * 3 * plane_sz + static_cast<ptrdiff_t>(y - 1) * fw + (xx - 1);
      float vn[27];
#pragma unroll
      for (int ci = 0; ci < 3; ++ci) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
          for (int s = 0; s < 3; ++s)
            vn[ci * 9 + r * 3 + s] = (ry[r] && cx[s]) ? __ldg(base + (ci * fplane + r * fw + s)) : 0.f;
        }
      }
      if (built > 0) {                                  // the previous tile's conv1_1 MMAs have read the buffer
        mbar_wait(i_empty, i_phase);
        i_phase ^= 1;
      }
      ++built;
      if (live) {                                       // k = ci*9 + 3r + s < 27, zero up to 32; hi / lo planes
#pragma unroll
        for (int chunk = 0; chunk < 4; ++chunk) {
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int k0 = chunk * 8 + 2 * t;
            split_pack2(k0 < 27 ? vn[k0 < 27 ? k0 : 0] : 0.f, k0 + 1 < 27 ? vn[k0 + 1 < 27 ? k0 + 1 : 0] : 0.f, hi[t], lo[t]);
          }
          *reinterpret_cast<uint4*>(smem_i + Cfg::offset(irow, chunk)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(smem_i + kS1Im2colPlane + Cfg::offset(irow, chunk)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      fence_proxy_async_smem();
      mbar_arrive(i_full);
    };
    const int first = static_cast<int>(blockIdx.x), stride = static_cast<int>(gridDim.x);
    for (int k = 0; k < 3; ++k)                         // operand rows of this CTA's first three tiles
      if (first + k * stride < p.total_tiles) build(first + k * stride);
    conv_epilogue_lean<64>(p, tmem_base, tfull_bar, tempty_bar, warp, lane, [&](int tile) {
      if (tile + 3 * stride < p.total_tiles) build(tile + 3 * stride);
    });
  } else {
    // ------------------------------------------------------------ stage-1 warps: conv1_1's epilogue (TMEM -> activation stage)
    // warps 10 .. 13 (TMEM lane quarters 2, 3, 0, 1): pixels 0 .. 127 = first M half; warps 14, 15 (quarters 2, 3):
    // pixels 128 .. 191 = lanes 64 .. 127 of the second M half (operand rows 192 .. 255)
    const int q = warp & 3;
    const int mh = warp >= 14 ? 1 : 0;
    const int pix = mh ? 128 + (q - 2) * 32 + lane : q * 32 + lane;     // halo pixel of this thread
    const bool live = pix < kS1HaloPx;
    const int hy = pix / kS1Pitch, hx = pix - hy * kS1Pitch;
    uint32_t c_phase = 0;
    int a_stage = 0;
    uint32_t a_phase = 0;
    const uint32_t taddr = tmem_c1 + mh * 128 + (static_cast<uint32_t>(q * 32) << 16);
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      int nb, tx, ty, img;
      decode_tile(p, tile, nb, tx, ty, img);
      const int y = ty * kTileH - 1 + hy, xx = tx * kTileW - 1 + hx;
      const bool inside = live && y >= 0 && y < p.h && xx >= 0 && xx < p.w;
      // ---- conv1_1 epilogue of this tile: TMEM -> bias / ReLU / zero padding -> split bf16 -> activation stage
      mbar_wait(&a_empty[a_stage], a_phase ^ 1);   // conv1_2's MMAs of two tiles ago have read this stage
      mbar_wait(c_full, c_phase);
      tc_fence_after();
      uint8_t* st = smem_a + a_stage * kS1AStage;
      uint32_t v[16], v2[16];
      tmem_ld16(taddr, v);                            // channels 0 .. 15: A_hi.B_hi + A_lo.B_hi
      tmem_ld16(taddr + 64, v2);                      //                   A_hi.B_lo
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {                // 16 channels at a time (register budget: 512 threads)
        float f[16];
        if (s1.b1) {
          const float4* bp = reinterpret_cast<const float4*>(s1.b1 + cc * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 b4 = __ldg(bp + j);
            f[4 * j] = b4.x, f[4 * j + 1] = b4.y, f[4 * j + 2] = b4.z, f[4 * j + 3] = b4.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = 0.f;
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          f[j] += __uint_as_float(v[j]);
          f[j] += __uint_as_float(v2[j]);
          f[j] = inside ? fmaxf(f[j], 0.f) : 0.f;     // ReLU; halo pixels outside the frame are conv1_2's zero padding
        }
        if (cc < 3) {                                 // the next 16 channels: in flight behind the split / stores
          tmem_ld16(taddr + (cc + 1) * 16, v);
          tmem_ld16(taddr + 64 + (cc + 1) * 16, v2);
        } else {                                      // every column read: conv1_1's accumulators may be overwritten
          tc_fence_before();
          mbar_arrive(c_empty);
        }
        if (live) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) split_pack2(f[8 * j + 2 * t], f[8 * j + 2 * t + 1], hi[t], lo[t]);
            const uint32_t off = sw128_offset(pix, cc * 2 + j);
            *reinterpret_cast<uint4*>(st + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(st + kS1APlane + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
      }
      fence_proxy_async_smem();
      mbar_arrive(&a_full[a_stage]);                   // conv1_2's MMAs may read the stage
      c_phase ^= 1;
      if (++a_stage == kS1AStages) {
        a_stage = 0;
        a_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace osvos

using namespace osvos;

extern "C" int osvos_stage1_fused(const osvos_stage1_args* a, osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(a != nullptr && a->x != nullptr && a->w1 != nullptr && a->w2_packed != nullptr);
  OSVOS_CHECK_ARG(a->n > 0 && a->h > 0 && a->w > 0 && a->h <= 65535 && a->n <= 65535);
  OSVOS_CHECK_ARG((a->y_hi != nullptr && a->y_lo != nullptr) || (a->pool_hi != nullptr && a->pool_lo != nullptr));
  OSVOS_CHECK_ARG((a->y_hi == nullptr) == (a->y_lo == nullptr) && (a->pool_hi == nullptr) == (a->pool_lo == nullptr));
  {
    const uintptr_t any = reinterpret_cast<uintptr_t>(a->y_hi) | reinterpret_cast<uintptr_t>(a->y_lo) |
                          reinterpret_cast<uintptr_t>(a->pool_hi) | reinterpret_cast<uintptr_t>(a->pool_lo);
    OSVOS_CHECK_ARG((any & 31) == 0);
    OSVOS_CHECK_ARG(((reinterpret_cast<uintptr_t>(a->b1) | reinterpret_cast<uintptr_t>(a->b2) |
                      reinterpret_cast<uintptr_t>(a->w2_packed)) & 15) == 0);
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  osvos_conv3x3_args c;
  memset(&c, 0, sizeof(c));
  c.w_packed = a->w2_packed;
  c.bias = a->b2;
  c.y_hi = a->y_hi;
  c.y_lo = a->y_lo;
  c.pool_hi = a->pool_hi;
  c.pool_lo = a->pool_lo;
  c.n = a->n, c.h = a->h, c.w = a->w, c.cin = 64, c.cout = 64;
  c.flags = OSVOS_FLAG_RELU;
  ConvParams p;
  fill_conv_params(p, &c, 64);
  CUtensorMap mw_hi, mw_lo;
  int rc = encode_weight_maps(&mw_hi, &mw_lo, a->w2_packed, 64, 64, 64, 1);
  if (rc) return rc;
  Stage1Params s1;
  s1.x = a->x;
  s1.w1 = a->w1;
  s1.b1 = a->b1;
  auto launch = [&](auto sw64) {
    constexpr bool SW64 = decltype(sw64)::value;
    return launch_persistent<conv_stage1_fused_kernel<SW64>>(p.total_tiles, kS1Threads, S1Cfg<SW64>::kSmem, stream, mw_hi,
                                                             mw_lo, s1, p);
  };
  OSVOS_CHECK_CUDA(env_int("OSVOS_S1_SW64", 1) != 0 ? launch(std::true_type{}) : launch(std::false_type{}));
  return OSVOS_OK;
}
