// side_prep: 3x3 convolution C -> 16 (no ReLU) + the fused 1x1 projections, with the NINE TAPS CONCATENATED ALONG N.
//
// With N = 16 a tcgen05.mma still costs its ~85-cycle floor, and the generic kernel issues one per (tap, K step, pass):
// the four side convolutions took 137 us of a 866 us frame at 9-14 % tensor activity.  Here the GEMM is turned around:
//   Y[p][tap*16 + co] = sum_ci X[p][ci] * W[tap][co][ci]        p = pixel of the UNSHIFTED halo patch
// i.e. ONE MMA of N = 144 per K step and pass (A = the 12 x 10-pixel halo patch of a 10 x 8 output tile, 120 of the 128
// GEMM rows; B = all nine 16 x 64 weight slabs of the chunk, one TMA box {64, 16, 9}), 9x fewer instructions.  The
// spatial shift moves to the epilogue: out[y][x][co] = sum_{r,s} Y[(y + r) * 10 + (x + s)][(3r + s) * 16 + co], done
// through a shared-memory exchange in three deterministic rounds (one tap row each).
//
// Replaces side_prep[i] (+ score_dsn[i] and this scale's slice of fuse as projections), reference
// networks/vgg_osvos.py:41,44,54 run at :67,69,72.  Same argument contract as osvos_conv3x3 with cout == 16.
//
// NCO = 2 - the FOLDED side branch (inference and training): side_prep has no ReLU, so side_prep followed by the two 1x1 projections
// (score_dsn, this scale's slice of fuse) is ONE linear 3x3 convolution C -> 2 whose weights are
// W'[o][ci][tap] = sum_co proj[o][co] * W_side[co][ci][tap] (osvos_fold_side_weights).  The same kernel then runs with
// N = 32 (18 used) instead of 144: 1/8 of the accumulator columns to exchange, 1/4.5 of the weight bytes to stream,
// a third less tensor time - the side branch was bound by exactly those (shared-memory bandwidth: the N = 144 MMA alone
// reads 120 B/clk of operands).  The backward of the folded form needs no features either (side_bwd_folded.cu); NCO = 16 stays
// for osvos_conv3x3 calls with cout == 16 (the literal side_prep op).
#include <string.h>

#include "conv_common.cuh"

namespace osvos {

constexpr int kSideTileW = 8, kSideTileH = 10;              // output tile
constexpr int kSideHaloW = 10, kSideHaloH = 12;             // 120 halo pixels = GEMM rows
constexpr int kSideThreads = 192;                           // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int kSideABox = kSideHaloW * kSideHaloH * 128;    // 15360 B
constexpr int kSideAPlane = 128 * 128;                      // the MMA reads 128 rows

// One launch serves up to four SCALES (inference: the folded side convolutions of stages 2-5 after the last trunk conv -
// one fill / drain and one launch instead of four, and the 21- and 84-tile scales no longer leave most SMs idle).  Tiles
// are numbered scale after scale, deepest (most channel chunks per tile) first, and dealt round-robin.
constexpr int kSideMaxScales = 4;
struct SideScale {
  const float* bias;
  float* y_f32;
  const float* proj_w;
  const float* proj_b;
  float* pq;
  int n, h, w, cin;
  int tiles_x, tiles_y, k_chunks;
  int tile_begin;    // first tile index of this scale
  int relu;
};
struct SideParams {
  SideScale sc[kSideMaxScales];
  int count;
  int total_tiles;
};
struct SideMaps {
  CUtensorMap x_hi[kSideMaxScales], x_lo[kSideMaxScales], w_hi[kSideMaxScales], w_lo[kSideMaxScales];
};

template <int PLANES, int NCO>
struct SideCfg {
  static_assert(NCO == 16 || NCO == 2, "16 side features, or the 2 folded projections");
  static constexpr int kN = NCO == 16 ? 144 : 32;             // MMA N: 9 taps x NCO columns (18 of the 32 used)
  static constexpr int kBBox = 9 * NCO * 128;                 // bytes the weight box of one chunk and plane delivers
  static constexpr int kBPlane = kN * 128;                    // 18432 / 4096 B: what the MMA reads (1 KiB multiple)
  static constexpr int kBStages = NCO == 16 ? 3 : 6;
  // activation ring: the folded kernel's step is ~600 cycles of MMA per 30 KiB chunk, far below the latency of the
  // chunk's TMA load - it needs loads of several chunks in flight (measured with 2 stages: 21 us for a 52 MB input)
  static constexpr int kAStages = NCO == 16 ? 2 : 4;
  static constexpr int kAStage = PLANES * kSideAPlane;
  static constexpr int kBStage = PLANES * kBPlane;
  // exchange buffer: NCO = 16: one tap row [s][co][halo px (128)] floats = 24 KiB;
  //                  NCO = 2: two buffers (alternating tiles) of [tap][halo px] float2 = 2 x 9 KiB
  static constexpr int kYBuf = NCO == 16 ? 3 * 16 * 128 * 4 : 2 * 9 * 128 * 8;
  static constexpr int kSmem = kAStages * kAStage + kBStages * kBStage + kYBuf + 1024 + 256;
};

__device__ __forceinline__ void side_decode(const SideParams& p, int tile, int& sc, int& tx, int& ty, int& img) {
  sc = 0;
  while (sc + 1 < p.count && tile >= p.sc[sc + 1].tile_begin) ++sc;
  const SideScale& L = p.sc[sc];
  const int local = tile - L.tile_begin;
  tx = local % L.tiles_x;
  const int t = local / L.tiles_x;
  ty = t % L.tiles_y;
  img = t / L.tiles_y;
}

template <int PLANES, int NCO>
__global__ void __launch_bounds__(kSideThreads, 1)
side_conv_kernel(const __grid_constant__ SideMaps maps, const __grid_constant__ SideParams p) {
  using Cfg = SideCfg<PLANES, NCO>;
  constexpr int kSideAStages = Cfg::kAStages, kSideBStages = Cfg::kBStages, kSideBPlane = Cfg::kBPlane, kSideN = Cfg::kN, kSideYBuf = Cfg::kYBuf;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem_a + kSideAStages * Cfg::kAStage;
  float* ybuf = reinterpret_cast<float*>(smem_b + kSideBStages * Cfg::kBStage);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(ybuf) + kSideYBuf);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + kSideAStages;
  uint64_t* b_full = a_empty + kSideAStages;
  uint64_t* b_empty = b_full + kSideBStages;
  uint64_t* tfull_bar = b_empty + kSideBStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.count; ++i) {
      tma_prefetch_desc(&maps.x_hi[i]);
      tma_prefetch_desc(&maps.w_hi[i]);
    }
    for (int i = 0; i < kSideAStages; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < kSideBStages; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);  // 2 accumulator stages x 144 columns (256-column stride)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();               // the previous kernel's activations are first read below (ptx.cuh)
  pdl_launch_dependents();

  if (warp == 0) {
    // ONE elected thread runs the whole producer loop (see conv3x3_halo.cu)
    if (elect_one()) {
    int a_stage = 0, b_stage = 0;
    uint32_t a_phase = 0, b_phase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      int sc, tx, ty, img;
      side_decode(p, tile, sc, tx, ty, img);
      const int k_chunks = p.sc[sc].k_chunks;
      const CUtensorMap* mx_hi = &maps.x_hi[sc];
      const CUtensorMap* mx_lo = &maps.x_lo[sc];
      const CUtensorMap* mw_hi = &maps.w_hi[sc];
      const CUtensorMap* mw_lo = &maps.w_lo[sc];
      for (int kc = 0; kc < k_chunks; ++kc) {
        mbar_wait(&a_empty[a_stage], a_phase ^ 1);
        mbar_wait(&b_empty[b_stage], b_phase ^ 1);
        {
          uint8_t* sa = smem_a + a_stage * Cfg::kAStage;
          uint8_t* sb = smem_b + b_stage * Cfg::kBStage;
          mbar_arrive_expect_tx(&a_full[a_stage], PLANES * kSideABox);
          tma_load_4d(mx_hi, &a_full[a_stage], sa, kc * 64, tx * kSideTileW - 1, ty * kSideTileH - 1, img);
          if (PLANES == 2)
            tma_load_4d(mx_lo, &a_full[a_stage], sa + kSideAPlane, kc * 64, tx * kSideTileW - 1,
                        ty * kSideTileH - 1, img);
          mbar_arrive_expect_tx(&b_full[b_stage], PLANES * Cfg::kBBox);
          tma_load_3d(mw_hi, &b_full[b_stage], sb, kc * 64, 0, 0);
          if (PLANES == 2) tma_load_3d(mw_lo, &b_full[b_stage], sb + kSideBPlane, kc * 64, 0, 0);
        }
        if (++a_stage == kSideAStages) {
          a_stage = 0;
          a_phase ^= 1;
        }
        if (++b_stage == kSideBStages) {
          b_stage = 0;
          b_phase ^= 1;
        }
      }
    }
    }
    __syncwarp();
  } else if (warp == 1) {
    // MMA issuer: one elected thread for the whole loop
    if (elect_one()) {
    constexpr uint32_t idesc = make_idesc_f16(128, kSideN, /*bf16=*/true);
    int a_stage = 0, b_stage = 0;
    uint32_t a_phase = 0, b_phase = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      mbar_wait(&tempty_bar[as], aph ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + as * 256;
      int sc, tx_, ty_, img_;
      side_decode(p, tile, sc, tx_, ty_, img_);
      const int k_chunks = p.sc[sc].k_chunks;
      for (int kc = 0; kc < k_chunks; ++kc) {
        mbar_wait(&a_full[a_stage], a_phase);
        mbar_wait(&b_full[b_stage], b_phase);
        tc_fence_after();
        {
          const uint32_t a_hi = smem_u32(smem_a + a_stage * Cfg::kAStage);
          const uint32_t b_hi = smem_u32(smem_b + b_stage * Cfg::kBStage);
          const uint64_t da_hi = make_smem_desc(a_hi, 16, 1024, kLayoutSW128);
          const uint64_t da_lo = make_smem_desc(a_hi + kSideAPlane, 16, 1024, kLayoutSW128);
          const uint64_t db_hi = make_smem_desc(b_hi, 16, 1024, kLayoutSW128);
          const uint64_t db_lo = make_smem_desc(b_hi + kSideBPlane, 16, 1024, kLayoutSW128);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t adv = static_cast<uint64_t>(k * 2);
            if (PLANES == 2) {
              umma_f16(tmem_d, da_lo + adv, db_hi + adv, idesc, (kc | k) != 0);
              umma_f16(tmem_d, da_hi + adv, db_lo + adv, idesc, 1);
              umma_f16(tmem_d, da_hi + adv, db_hi + adv, idesc, 1);
            } else {
              umma_f16(tmem_d, da_hi + adv, db_hi + adv, idesc, (kc | k) != 0);
            }
          }
          umma_commit(&a_empty[a_stage]);
          umma_commit(&b_empty[b_stage]);
          if (kc == k_chunks - 1) umma_commit(&tfull_bar[as]);
        }
        if (++a_stage == kSideAStages) {
          a_stage = 0;
          a_phase ^= 1;
        }
        if (++b_stage == kSideBStages) {
          b_stage = 0;
          b_phase ^= 1;
        }
      }
    }
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- epilogue: shift-add through shared memory
    const int q = warp & 3;
    const int row = q * 32 + lane;                 // halo pixel index (valid < 120) / output thread index (< 80)
    const int oy = row / kSideTileW, ox = row % kSideTileW;   // as an OUTPUT pixel of the tile (row < 80)
    int it = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      int sc, tx, ty, img;
      side_decode(p, tile, sc, tx, ty, img);
      const SideScale& L = p.sc[sc];
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      mbar_wait(&tfull_bar[as], aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + as * 256 + (static_cast<uint32_t>(q * 32) << 16);
      if constexpr (NCO == 2) {
        // folded projections: column 2 * tap + o of halo pixel `row`.  One read, accumulator handed back at once, one
        // exchange through the buffer of this tile's parity (a single barrier per tile), nine float2 gathers.
        uint32_t v[32];
        tmem_ld32(taddr, v);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&tempty_bar[as]);
        float2* yb = reinterpret_cast<float2*>(ybuf) + (it & 1) * 9 * 128;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap)
          yb[tap * 128 + row] = make_float2(__uint_as_float(v[2 * tap]), __uint_as_float(v[2 * tap + 1]));
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const int y = ty * kSideTileH + oy, x = tx * kSideTileW + ox;
        if (row < kSideTileW * kSideTileH && y < L.h && x < L.w) {
          float sp = L.bias ? __ldg(L.bias) : 0.f, sq = L.bias ? __ldg(L.bias + 1) : 0.f;
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            const float2 t = yb[tap * 128 + (oy + tap / 3) * kSideHaloW + ox + tap % 3];
            sp += t.x;
            sq += t.y;
          }
          const size_t pix = (static_cast<size_t>(img) * L.h + y) * L.w + x;
          *reinterpret_cast<float2*>(L.pq + pix * 2) = make_float2(sp, sq);
        }
        continue;
      }
      float acc[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[j] = L.bias ? __ldg(L.bias + j) : 0.f;
#pragma unroll 1
      for (int r = 0; r < 3; ++r) {
        // (1) every halo-pixel thread publishes its three taps of row r: ybuf[s][co][pixel]
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          uint32_t v[16];
          tmem_ld16(taddr + (r * 3 + s) * 16, v);
          tmem_ld_wait();
#pragma unroll
          for (int co = 0; co < 16; ++co) ybuf[(s * 16 + co) * 128 + row] = __uint_as_float(v[co]);
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        // (2) output-pixel threads gather: halo pixel (oy + r, ox + s)
        if (row < kSideTileW * kSideTileH) {
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            const int src = (oy + r) * kSideHaloW + ox + s;
#pragma unroll
            for (int co = 0; co < 16; ++co) acc[co] += ybuf[(s * 16 + co) * 128 + src];
          }
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      tc_fence_before();
      mbar_arrive(&tempty_bar[as]);
      const int y = ty * kSideTileH + oy, x = tx * kSideTileW + ox;
      if (row < kSideTileW * kSideTileH && y < L.h && x < L.w) {
        const size_t pix = (static_cast<size_t>(img) * L.h + y) * L.w + x;
        if (L.relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[j] = fmaxf(acc[j], 0.f);
        }
        if (L.y_f32) {
          float4* dst = reinterpret_cast<float4*>(L.y_f32 + pix * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) dst[j] = make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
        }
        if (L.pq) {
          float sp = L.proj_b ? __ldg(L.proj_b) : 0.f, sq = 0.f;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            sp = fmaf(acc[j], __ldg(L.proj_w + j), sp);
            sq = fmaf(acc[j], __ldg(L.proj_w + 16 + j), sq);
          }
          *reinterpret_cast<float2*>(L.pq + pix * 2) = make_float2(sp, sq);
        }
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

template <int PLANES, int NCO>
static int launch_side(const osvos_conv3x3_args* const* args, int count, cudaStream_t stream) {
  using Cfg = SideCfg<PLANES, NCO>;
  SideParams p;
  SideMaps maps;
  memset(&p, 0, sizeof(p));
  p.count = count;
  int total = 0;
  for (int k = 0; k < count; ++k) {
    const osvos_conv3x3_args* a = args[k];
    SideScale& L = p.sc[k];
    L.bias = a->bias;
    L.y_f32 = a->y_f32;
    L.proj_w = a->proj_w;
    L.proj_b = a->proj_b;
    L.pq = a->pq;
    L.n = a->n;
    L.h = a->h;
    L.w = a->w;
    L.cin = a->cin;
    L.tiles_x = (a->w + kSideTileW - 1) / kSideTileW;
    L.tiles_y = (a->h + kSideTileH - 1) / kSideTileH;
    L.k_chunks = a->cin / 64;
    L.relu = (a->flags & OSVOS_FLAG_RELU) ? 1 : 0;
    L.tile_begin = total;
    total += L.tiles_x * L.tiles_y * a->n;
    int rc = encode_act_maps(&maps.x_hi[k], &maps.x_lo[k], a->x_hi, PLANES == 2 ? a->x_lo : nullptr, a->n, a->h, a->w,
                             a->cin, kSideHaloW, kSideHaloH);
    if (rc) return rc;
    rc = encode_weight_maps(&maps.w_hi[k], &maps.w_lo[k], a->w_packed, NCO, a->cin, NCO, 9);   // all nine taps
    if (rc) return rc;
  }
  for (int k = count; k < kSideMaxScales; ++k) {   // unused slots: valid descriptors (never dereferenced)
    maps.x_hi[k] = maps.x_hi[0];
    maps.x_lo[k] = maps.x_lo[0];
    maps.w_hi[k] = maps.w_hi[0];
    maps.w_lo[k] = maps.w_lo[0];
  }
  p.total_tiles = total;
  OSVOS_CHECK_CUDA((launch_persistent<side_conv_kernel<PLANES, NCO>>(p.total_tiles, kSideThreads, Cfg::kSmem, stream, maps,
                                                                     p)));
  return OSVOS_OK;
}

int side_conv_dispatch(const osvos_conv3x3_args* a, cudaStream_t stream) {
  const osvos_conv3x3_args* one[1] = {a};
  if (a->cout == 2)   // folded projections (osvos_fold_side_weights): pq only
    return (a->flags & OSVOS_FLAG_FAST) ? launch_side<1, 2>(one, 1, stream) : launch_side<2, 2>(one, 1, stream);
  return (a->flags & OSVOS_FLAG_FAST) ? launch_side<1, 16>(one, 1, stream) : launch_side<2, 16>(one, 1, stream);
}

// Folded side convolutions of several scales in one launch; `args` sorted deepest (most input channels) first.
int side_conv_multi_dispatch(const osvos_conv3x3_args* const* args, int count, cudaStream_t stream) {
  const bool fast = (args[0]->flags & OSVOS_FLAG_FAST) != 0;
  return fast ? launch_side<1, 2>(args, count, stream) : launch_side<2, 2>(args, count, stream);
}

}  // namespace osvos
