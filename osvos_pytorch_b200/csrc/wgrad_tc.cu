// Weight gradient of the 3x3 convolutions as a tcgen05 GEMM whose reduction
// dimension is the PIXEL axis:
//
//   ws[tap][m][n] += sum_px P[px (+tap)][m] * Q[px (+tap)][n]
//
// P = dZ (gradient of the conv output, unshifted, m = co) and Q = the layer's input
// activation shifted by the tap (n = ci).  (side_prep's weight gradient is not a GEMM
// of this shape any more: side_bwd_folded.cu.)  Both operands are
// NHWC acts, i.e. the reduction index (pixel) is the strided one: they are
// "MN-major" UMMA operands.  A K block is a patch of 8 x 8 pixels; its TMA box
// {64 ch, 8 px, 8 rows, 1} lands as 64 rows x 128 B (SWIZZLE_128B), which is the
// canonical MN-major SW128 atom layout (64 MN elements x 8 K rows per atom,
// SBO = 1024 B between K groups, LBO = 8192 B between 64-wide MN atoms).
// Out-of-image pixels are zero-filled by TMA: they are both the conv padding of
// the shifted operand and the ragged-edge mask of the unshifted one.
//
// Work item = (m block of 128, n block, tap, pixel-range split); the fp32 TMEM
// accumulator is flushed with vector atomics (red.global.add.v4.f32) into the
// zero-initialised workspace, which a small kernel then transposes into the
// OIHW gradient.  Warps 0 and 6 are the TMA producers of P and Q, warp 1 the MMA
// issuer, warps 2-5 the epilogue; mbarrier rings as in conv3x3_halo.cu.
//
// Replaces autograd's weight gradient of nn.Conv2d(k=3, p=1)
// (reference networks/vgg_osvos.py:41,142; backward triggered at train_online.py:141).
#include <string.h>

#include "common.cuh"
#include "ptx.cuh"

namespace osvos {

constexpr int kWgThreads = 224;   // warp 0: P producer, 1: MMA, 2-5: epilogue, 6: Q producer
constexpr int kWgPatchW = 8, kWgPatchH = 8;
constexpr int kWgBlockK = 64;                  // pixels per K block
constexpr int kWgBoxBytes = kWgBlockK * 128;   // 8 KiB: 64 pixels x 64 channels of bf16

struct WgradParams {
  float* ws;  // [9][m_total][n_total]
  int n_img, h, w;
  int m_total, n_total, m_valid;
  int m_blocks, n_blocks, splits;
  int patches_x, patches_y, patches_total, patches_per_split;
  int total_items;
  int tap_pairs;  // 1: Q has 64 channels and the two 64-wide N atoms of a 128-wide item are TWO TAPS (2g, 2g+1)
  int tap_rows;   // 1: P AND Q have 64 channels (conv1_2): an item is one tap ROW - see launch_wgrad
  int tap_items;  // 9, 5 tap groups in tap_pairs mode, or 3 tap rows in tap_rows mode
};

template <int BLOCK_N, int PLANES>
struct WgCfg {
  static constexpr int kPBytes = 2 * kWgBoxBytes;               // 128 m
  static constexpr int kQBytes = (BLOCK_N / 64) * kWgBoxBytes;  // BLOCK_N n
  static constexpr int kStageBytes = PLANES * (kPBytes + kQBytes);
  static constexpr int kStagesRaw = (212 * 1024) / kStageBytes;
  static constexpr int kStages = kStagesRaw > 8 ? 8 : kStagesRaw;
  // Exact mode: N-concatenated split-Q.  The hi and lo planes of the Q tile are contiguous (uniform LBO between
  // the 64-wide MN atoms), so one tcgen05.mma of N = 2 * BLOCK_N yields [P_hi.Q_hi | P_hi.Q_lo]; with P_lo.Q_hi
  // that is 2 instructions per K step instead of 3 (see conv3x3_halo.cu).  The epilogue adds the two halves.
  static constexpr bool kSplitAcc = (PLANES == 2) && (BLOCK_N <= 128);
  static constexpr int kAccCols = kSplitAcc ? 2 * BLOCK_N : BLOCK_N;
  static constexpr int kTmemCols = 2 * kAccCols < 32 ? 32 : 2 * kAccCols;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 256;
  // descriptors are formed by adding (bytes >> 4) to a base descriptor (see conv3x3_halo.cu): stay inside the field
  static_assert(kSmemBytes <= 227 * 1024 && kSmemBytes + 8192 < (1 << 18), "shared memory / descriptor address field");
};

__device__ __forceinline__ void wg_decode_item(const WgradParams& p, int item, int& mb, int& nb, int& tap, int& split) {
  nb = item % p.n_blocks;
  int t = item / p.n_blocks;
  mb = t % p.m_blocks;
  t /= p.m_blocks;
  tap = t % p.tap_items;   // tap index, or tap-group index in tap_pairs mode
  split = t / p.tap_items;
}

template <int BLOCK_N, int PLANES>
__global__ void __launch_bounds__(kWgThreads, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_p_hi, const __grid_constant__ CUtensorMap map_p_lo,
                const __grid_constant__ CUtensorMap map_q_hi, const __grid_constant__ CUtensorMap map_q_lo,
                const WgradParams p) {
  using Cfg = WgCfg<BLOCK_N, PLANES>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::kStageBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kStages;
  uint64_t* tfull_bar = bars + 2 * kStages;
  uint64_t* tempty_bar = bars + 2 * kStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_p_hi);
    tma_prefetch_desc(&map_q_hi);
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 2);   // one arrive.expect_tx from each of the two producer warps
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();               // dz / x come from the previous kernels of the stream (ptx.cuh)
  pdl_launch_dependents();

  if (warp == 0 || warp == 6) {
    // two producer warps (P operand: warp 0, Q operand: warp 6) halve the per-K-block TMA issue time.  ONE elected
    // thread per warp runs the whole loop (no per-step ELECT / reconvergence - see conv3x3_halo.cu); the patch
    // coordinates advance incrementally instead of by two integer divisions per K block.
    if (elect_one()) {
      const bool load_p = (warp == 0);
      int stage = 0;
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < p.total_items; item += gridDim.x) {
        int mb, nb, tap, split;
        wg_decode_item(p, item, mb, nb, tap, split);
        const int tap0 = p.tap_pairs ? 2 * tap : tap;
        const int tap1 = (p.tap_pairs && tap0 + 1 < 9) ? tap0 + 1 : tap0;   // second N atom (tap 8 is alone: repeated, unused)
        const int dy = tap0 / 3 - 1, dx = tap0 % 3 - 1;
        const int dy1 = tap1 / 3 - 1, dx1 = tap1 % 3 - 1;
        const int qdy = dy, qdx = dx;      // Q is the shifted operand (zero-filled outside the image = conv padding)
        const int pb = split * p.patches_per_split;
        int pe = pb + p.patches_per_split;
        if (pe > p.patches_total) pe = p.patches_total;
        int px = pb % p.patches_x;
        int py = (pb / p.patches_x) % p.patches_y;
        int img = pb / (p.patches_x * p.patches_y);
        const int c_p = mb * 128, c_q = nb * BLOCK_N;
        for (int patch = pb; patch < pe; ++patch) {
          const int x0 = px * kWgPatchW, y0 = py * kWgPatchH;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* st = smem + stage * Cfg::kStageBytes;
          if (load_p) {
            mbar_arrive_expect_tx(&full_bar[stage], PLANES * Cfg::kPBytes);
#pragma unroll
            for (int pl = 0; pl < PLANES; ++pl) {
              const CUtensorMap* mp = pl == 0 ? &map_p_hi : &map_p_lo;
              uint8_t* sp = st + pl * Cfg::kPBytes;
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                if (p.tap_rows)   // M atom j = the single 64-channel block of dz shifted by (0, +j)
                  tma_load_4d(mp, &full_bar[stage], sp + j * kWgBoxBytes, 0, x0 + j, y0, img);
                else
                  tma_load_4d(mp, &full_bar[stage], sp + j * kWgBoxBytes, c_p + j * 64, x0, y0, img);
              }
            }
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], PLANES * Cfg::kQBytes);
#pragma unroll
            for (int pl = 0; pl < PLANES; ++pl) {
              const CUtensorMap* mq = pl == 0 ? &map_q_hi : &map_q_lo;
              uint8_t* sq = st + PLANES * Cfg::kPBytes + pl * Cfg::kQBytes;
#pragma unroll
              for (int j = 0; j < BLOCK_N / 64; ++j) {
                if (p.tap_rows)    // N atom j = the single 64-channel block of x shifted by (row - 1, +j)
                  tma_load_4d(mq, &full_bar[stage], sq + j * kWgBoxBytes, 0, x0 + j, y0 + tap - 1, img);
                else if (p.tap_pairs)   // atom j = tap (2g + j) of the single 64-channel block
                  tma_load_4d(mq, &full_bar[stage], sq + j * kWgBoxBytes, 0, x0 + (j ? dx1 : dx), y0 + (j ? dy1 : dy), img);
                else
                  tma_load_4d(mq, &full_bar[stage], sq + j * kWgBoxBytes, c_q + j * 64, x0 + qdx, y0 + qdy, img);
              }
            }
          }
          if (++px == p.patches_x) {
            px = 0;
            if (++py == p.patches_y) {
              py = 0;
              ++img;
            }
          }
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // MMA issuer: one elected thread, descriptors formed by adding the stage offset to a constant template
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_f16(128, BLOCK_N, true, /*a_mn=*/true, /*b_mn=*/true);
      constexpr uint32_t idesc2 = make_idesc_f16(128, Cfg::kAccCols, true, /*a_mn=*/true, /*b_mn=*/true);
      // MN-major SW128: LBO = bytes between 64-wide MN atoms, SBO = bytes between 8-row K groups
      constexpr uint64_t kDesc = (static_cast<uint64_t>(kWgBoxBytes >> 4) << 16) | (static_cast<uint64_t>(1024 >> 4) << 32) |
                                 (1ull << 46) | (static_cast<uint64_t>(kLayoutSW128) << 61);
      constexpr uint32_t kQOff = (PLANES * Cfg::kPBytes) >> 4, kPLo = Cfg::kPBytes >> 4, kQLo = Cfg::kQBytes >> 4;
      const uint32_t smem_base = smem_u32(smem);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int item = blockIdx.x; item < p.total_items; item += gridDim.x, ++it) {
        int mb, nb, tap, split;
        wg_decode_item(p, item, mb, nb, tap, split);
        const int pb = split * p.patches_per_split;
        int pe = pb + p.patches_per_split;
        if (pe > p.patches_total) pe = p.patches_total;
        const int as = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait(&tempty_bar[as], aph ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * Cfg::kAccCols;
        for (int patch = pb; patch < pe; ++patch) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t dp_hi = kDesc | static_cast<uint64_t>((smem_base + stage * Cfg::kStageBytes) >> 4);
          const uint64_t dq_hi = dp_hi + kQOff;
          const uint64_t dp_lo = dp_hi + kPLo;
          const uint64_t dq_lo = dq_hi + kQLo;
#pragma unroll
          for (int k = 0; k < kWgBlockK / 16; ++k) {
            const uint32_t adv = static_cast<uint32_t>(k * (2048 >> 4));  // 16 pixel rows x 128 B
            const uint32_t acc = (k != 0) ? 1u : (patch != pb ? 1u : 0u);
            if (Cfg::kSplitAcc) {
              umma_f16(tmem_d, dp_hi + adv, dq_hi + adv, idesc2, acc);   // [P_hi.Q_hi | P_hi.Q_lo]
              umma_f16(tmem_d, dp_lo + adv, dq_hi + adv, idesc, 1);      // + P_lo.Q_hi into the first half
            } else if (PLANES == 2) {
              umma_f16(tmem_d, dp_lo + adv, dq_hi + adv, idesc, acc);
              umma_f16(tmem_d, dp_hi + adv, dq_lo + adv, idesc, 1);
              umma_f16(tmem_d, dp_hi + adv, dq_hi + adv, idesc, 1);
            } else {
              umma_f16(tmem_d, dp_hi + adv, dq_hi + adv, idesc, acc);
            }
          }
          umma_commit(&empty_bar[stage]);
          if (patch == pe - 1) umma_commit(&tfull_bar[as]);
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 2 && warp < 6) {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    int it = 0;
    for (int item = blockIdx.x; item < p.total_items; item += gridDim.x, ++it) {
      int mb, nb, tap, split;
      wg_decode_item(p, item, mb, nb, tap, split);
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const int m = mb * 128 + row;
      mbar_wait(&tfull_bar[as], aph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + as * Cfg::kAccCols + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
      for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
        // destination of this 32-column chunk: channel block nb, or (tap_pairs) tap 2g + c0/64 of the 64 channels, or
        // (tap_rows) the tap = shift of the N atom minus shift of the M atom: (M0,N0) -> s = 1, (M0,N1) -> s = 2,
        // (M1,N0) -> s = 0, (M1,N1) -> s = 1 again (discarded)
        int tap_c = p.tap_pairs ? 2 * tap + (c0 >> 6) : tap;
        bool chunk_ok = tap_c < 9;
        int m_out = m;
        if (p.tap_rows) {
          const int pj = row >> 6, qj = c0 >> 6;
          chunk_ok = !(pj && qj);
          tap_c = 3 * tap + (pj ? 0 : 1 + qj);
          m_out = row & 63;
        }
        float* dst = p.ws + (static_cast<size_t>(chunk_ok ? tap_c : 0) * p.m_total + m_out) * p.n_total +
                     ((p.tap_pairs || p.tap_rows) ? -(c0 & ~63) : nb * BLOCK_N);
        uint32_t v[32], v2[32];
        tmem_ld32(taddr + c0, v);
        if (Cfg::kSplitAcc) tmem_ld32(taddr + BLOCK_N + c0, v2);
        tmem_ld_wait();
        if ((m < p.m_valid || p.tap_rows) && chunk_ok) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float4 val = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                     __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            if (Cfg::kSplitAcc) {
              val.x += __uint_as_float(v2[4 * j]);
              val.y += __uint_as_float(v2[4 * j + 1]);
              val.z += __uint_as_float(v2[4 * j + 2]);
              val.w += __uint_as_float(v2[4 * j + 3]);
            }
            atomicAdd(reinterpret_cast<float4*>(dst + c0 + 4 * j), val);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty_bar[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ws[tap][co][ci] -> OIHW gradient (the immediate, non-deferred form of one layer).
__global__ void wgrad_finish_kernel(const float* __restrict__ ws, float* __restrict__ dw, int cout, int cin, int ld_a,
                                    int ld_b) {
  const int total = cout * cin * 9;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int tap = i % 9;
    const int ci = (i / 9) % cin;
    const int co = i / (9 * cin);
    dw[i] = ws[(static_cast<size_t>(tap) * ld_a + co) * ld_b + ci];
  }
}

// Deferred finish of many layers in one launch.  A work item is one output row (co) x 64 input channels x 9 taps
// = 576 contiguous OIHW floats: the nine workspace rows are read coalesced (256 B each), transposed through shared
// memory and written coalesced.
struct FinishLayer {
  const float* ws;
  float* dw;
  int cout, cin, ld_a, ld_b, accumulate;
  float scale;
  int items;
};
struct FinishTable {
  FinishLayer layer[OSVOS_WGRAD_FINISH_MAX];
  int count;
  int total_items;
};
constexpr int kFinishThreads = 192;
constexpr int kFinishChunk = 576;

__global__ void __launch_bounds__(kFinishThreads)
wgrad_finish_multi_kernel(const __grid_constant__ FinishTable t) {
  __shared__ __align__(16) float tile[9][68];
  // each block takes a contiguous range of items, so the layer index only moves forward
  const int per = (t.total_items + gridDim.x - 1) / gridDim.x;
  const int begin = blockIdx.x * per, end = min(begin + per, t.total_items);
  int li = 0, base = 0;
  for (int work = begin; work < end; ++work) {
    while (work - base >= t.layer[li].items) {
      base += t.layer[li].items;
      ++li;
    }
    const FinishLayer& L = t.layer[li];
    const int item = work - base;
    const int chunks = L.cin / 64;
    const int co = item / chunks, ci0 = (item - co * chunks) * 64;
    __syncthreads();   // previous item's readers of `tile` are done
    if (threadIdx.x < 144) {   // 9 taps x 16 float4
      const int tap = threadIdx.x >> 4, c4 = threadIdx.x & 15;
      const float4 v = __ldg(reinterpret_cast<const float4*>(L.ws + (static_cast<size_t>(tap) * L.ld_a + co) * L.ld_b + ci0) + c4);
      *reinterpret_cast<float4*>(&tile[tap][c4 * 4]) = v;
    }
    __syncthreads();
    float* out = L.dw + (static_cast<size_t>(co) * L.cin + ci0) * 9;
    if ((reinterpret_cast<uintptr_t>(out) & 15) == 0) {
      if (threadIdx.x < 144) {   // 576 contiguous floats = 144 float4
        const int e = threadIdx.x * 4;
        float4 v;
        v.x = tile[e % 9][e / 9] * L.scale;
        v.y = tile[(e + 1) % 9][(e + 1) / 9] * L.scale;
        v.z = tile[(e + 2) % 9][(e + 2) / 9] * L.scale;
        v.w = tile[(e + 3) % 9][(e + 3) / 9] * L.scale;
        float4* o = reinterpret_cast<float4*>(out) + threadIdx.x;
        if (L.accumulate) {
          const float4 g = *o;
          v.x += g.x, v.y += g.y, v.z += g.z, v.w += g.w;
        }
        *o = v;
      }
    } else {
      for (int i = threadIdx.x; i < kFinishChunk; i += kFinishThreads) {
        const float v = tile[i % 9][i / 9] * L.scale;
        out[i] = L.accumulate ? out[i] + v : v;
      }
    }
  }
}

// The switches of launch_wgrad: OSVOS_WGRAD_ROWS, OSVOS_WGRAD_SPLITS (runtime.cu).
struct WgradSwitches {
  bool rows, legacy_split;
};
static WgradSwitches wgrad_switches() {
  return WgradSwitches{env_int("OSVOS_WGRAD_ROWS", 1) != 0, env_is("OSVOS_WGRAD_SPLITS", "legacy")};
}

// The work decomposition of one launch: every WgradParams field that is not a pointer or an image dimension, and the
// persistent grid.  One pure function of the arguments, the SM count and the switches, so that
// osvos_conv3x3_wgrad_plan reports exactly what osvos_conv3x3_wgrad runs.  Returns OSVOS_ERR_UNSUPPORTED for a dz
// channel count the kernel cannot tile.
static int plan_wgrad(const osvos_wgrad_args* a, int block_n, int sms, const WgradSwitches& sw, WgradParams& p, int& grid) {
  const int cp = a->dz_channels;   // channels of the P tensor
  const int cq = a->cin;           // channels of the Q tensor
  p.n_img = a->n;
  p.h = a->h;
  p.w = a->w;
  p.m_total = (cp + 127) / 128 * 128;
  if (p.m_total != cp && cp != 64) return OSVOS_ERR_UNSUPPORTED;
  p.m_total = cp;  // rows actually stored in the workspace
  p.m_valid = cp;
  p.n_total = cq;
  p.m_blocks = (cp + 127) / 128;
  // Cin = 64 trunk layers (conv1_2, conv2_1): the 128-wide item holds two TAPS of the single 64-channel block, which
  // halves the number of tcgen05.mma (the ~85-cycle instruction floor makes N = 64 items twice as expensive per flop)
  // Cin = Cout = 64 (conv1_2): an item is a tap ROW r.  M = [dz | dz shifted by (0,+1)], N = [x shifted by (r-1, 0) |
  // x shifted by (r-1, +1)]: the four 64 x 64 quadrants are the taps s = 1, 2, 0 and 1 again - three of four useful
  // instead of the two of four of tap pairs under a half-empty M (a tcgen05.mma costs max(M, 128) rows either way).
  // Exact at the borders: the terms dz[u] x[u + (., -1)] the shifted M atom cannot reach (u.x = 0) multiply the zero
  // padding of x, and everything out of the image is zero-filled by TMA on both operands.
  p.tap_rows = (sw.rows && cq == 64 && cp == 64 && block_n == 128) ? 1 : 0;
  p.tap_pairs = (cq == 64 && block_n == 128 && !p.tap_rows) ? 1 : 0;
  p.tap_items = p.tap_rows ? 3 : p.tap_pairs ? 5 : 9;
  p.n_blocks = (p.tap_pairs || p.tap_rows) ? 1 : cq / block_n;
  p.patches_x = (a->w + kWgPatchW - 1) / kWgPatchW;
  p.patches_y = (a->h + kWgPatchH - 1) / kWgPatchH;
  p.patches_total = p.patches_x * p.patches_y * a->n;
  const int tiles = p.m_blocks * p.n_blocks * p.tap_items;
  // Pixel-range splits: items are dealt round-robin to the persistent CTAs, so the kernel lasts as long as the CTA with
  // the most items - ROUNDS x K blocks per item.  Pick the split count that minimises that (plus ~2 K-block times per
  // item for the accumulator flush that is not hidden behind the next item's MMAs).  The first rule, ceil(2 SMs /
  // tiles), landed just ABOVE two full rounds for most layers (297 items on 148 CTAs: a third round for one item,
  // 67 % of the tensor time) - profiles/r02l_*.
  const int max_splits = (p.patches_total + 3) / 4;
  int splits = 1;
  if (sw.legacy_split) {
    splits = (2 * sms + tiles - 1) / tiles;
  } else {
    long best = -1;
    const int s_hi = 4 * sms / tiles + 1;
    for (int s = 1; s <= s_hi && s <= max_splits; ++s) {
      const long pps = (p.patches_total + s - 1) / s;
      const long se = (p.patches_total + pps - 1) / pps;
      const long rounds = (static_cast<long>(tiles) * se + sms - 1) / sms;
      const long cost = rounds * (pps + 2) + 4;
      if (best < 0 || cost < best) {
        best = cost;
        splits = s;
      }
    }
  }
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  p.patches_per_split = (p.patches_total + splits - 1) / splits;
  p.splits = (p.patches_total + p.patches_per_split - 1) / p.patches_per_split;
  p.total_items = tiles * p.splits;
  grid = persistent_grid(p.total_items, sms);
  return OSVOS_OK;
}

template <int BLOCK_N, int PLANES>
static int launch_wgrad(const osvos_wgrad_args* a, cudaStream_t stream) {
  using Cfg = WgCfg<BLOCK_N, PLANES>;
  WgradParams p;
  int grid = 0;
  int rc = plan_wgrad(a, BLOCK_N, device_sm_count(), wgrad_switches(), p, grid);
  if (rc) return rc;
  p.ws = a->workspace;

  // operands: P = dz (dz_channels), Q = the layer's input x (cin)
  CUtensorMap mp_hi, mp_lo, mq_hi, mq_lo;
  rc = encode_act_maps(&mp_hi, &mp_lo, a->dz_hi, PLANES == 2 ? a->dz_lo : nullptr, a->n, a->h, a->w, a->dz_channels,
                       kWgPatchW, kWgPatchH);
  if (rc) return rc;
  rc = encode_act_maps(&mq_hi, &mq_lo, a->x_hi, PLANES == 2 ? a->x_lo : nullptr, a->n, a->h, a->w, a->cin, kWgPatchW,
                       kWgPatchH);
  if (rc) return rc;

  constexpr auto kern = wgrad_tc_kernel<BLOCK_N, PLANES>;
  if (a->flags & OSVOS_FLAG_DEFER_FINISH) {
    OSVOS_CHECK_CUDA((launch_persistent<kern>(p.total_items, kWgThreads, Cfg::kSmemBytes, stream, mp_hi, mp_lo, mq_hi,
                                              mq_lo, p)));
    return OSVOS_OK;
  }
  // immediate form: the memset is this kernel's stream predecessor, so a plain launch
  const size_t ws_bytes = static_cast<size_t>(9) * p.m_total * p.n_total * sizeof(float);
  OSVOS_CHECK_CUDA(cudaMemsetAsync(a->workspace, 0, ws_bytes, stream));
  OSVOS_CHECK_CUDA(ensure_dynamic_smem<kern>(Cfg::kSmemBytes));
  kern<<<grid, kWgThreads, Cfg::kSmemBytes, stream>>>(mp_hi, mp_lo, mq_hi, mq_lo, p);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  const int total = a->cout * a->cin * 9;
  wgrad_finish_kernel<<<(total + 255) / 256, 256, 0, stream>>>(a->workspace, a->dw, a->cout, a->cin, p.m_total, p.n_total);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

}  // namespace osvos

using namespace osvos;

extern "C" size_t osvos_wgrad_workspace_bytes(int cout_or_padded, int cin) {
  return static_cast<size_t>(9) * cout_or_padded * cin * sizeof(float);
}

extern "C" int osvos_wgrad_finish(const osvos_wgrad_finish_item* items, int count, osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(items != nullptr && count > 0 && count <= OSVOS_WGRAD_FINISH_MAX);
  FinishTable t;
  t.count = count;
  long long total_items = 0;
  for (int i = 0; i < count; ++i) {
    const osvos_wgrad_finish_item& it = items[i];
    OSVOS_CHECK_ARG(it.workspace != nullptr && it.dw != nullptr && it.cout > 0 && it.cin > 0 && it.cin % 64 == 0);
    OSVOS_CHECK_ARG(it.dz_channels % 64 == 0 && it.cout == it.dz_channels);
    FinishLayer& L = t.layer[i];
    L.ws = it.workspace;
    L.dw = it.dw;
    L.cout = it.cout;
    L.cin = it.cin;
    L.ld_a = it.dz_channels;
    L.ld_b = it.cin;
    L.accumulate = it.accumulate ? 1 : 0;
    L.scale = it.scale;
    L.items = it.cout * (it.cin / 64);
    total_items += L.items;
  }
  OSVOS_CHECK_ARG(total_items < (1ll << 31));
  t.total_items = static_cast<int>(total_items);
  const long long cap = static_cast<long long>(device_sm_count()) * 10;   // 10 x 192 threads resident per SM
  const unsigned grid = static_cast<unsigned>(total_items < cap ? total_items : cap);
  wgrad_finish_multi_kernel<<<grid, kFinishThreads, 0, static_cast<cudaStream_t>(stream_)>>>(t);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

static int check_wgrad_args(const osvos_wgrad_args* a) {
  OSVOS_CHECK_ARG(a != nullptr && a->x_hi != nullptr && a->dz_hi != nullptr && a->workspace != nullptr);
  OSVOS_CHECK_ARG(a->dw != nullptr || (a->flags & OSVOS_FLAG_DEFER_FINISH));
  OSVOS_CHECK_ARG(a->n > 0 && a->h > 0 && a->w > 0 && a->cin % 64 == 0 && a->dz_channels % 64 == 0);
  OSVOS_CHECK_ARG(a->cout == a->dz_channels);
  OSVOS_CHECK_ARG((a->flags & OSVOS_FLAG_FAST) || (a->x_lo != nullptr && a->dz_lo != nullptr));
  OSVOS_CHECK_ARG(a->cin % 128 == 0 || a->cin == 64);     // Cin = 64: tap-pair / tap-row modes of the 128-wide kernel
  return OSVOS_OK;
}

extern "C" int osvos_conv3x3_wgrad(const osvos_wgrad_args* a, osvos_stream_t stream_) {
  int rc = check_wgrad_args(a);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool fast = (a->flags & OSVOS_FLAG_FAST) != 0;
  return fast ? launch_wgrad<128, 1>(a, stream) : launch_wgrad<128, 2>(a, stream);
}

extern "C" int osvos_conv3x3_wgrad_plan(const osvos_wgrad_args* a, osvos_launch_plan* plan) {
  int rc = check_wgrad_args(a);
  if (rc) return rc;
  OSVOS_CHECK_ARG(plan != nullptr);
  const bool fast = (a->flags & OSVOS_FLAG_FAST) != 0;
  constexpr int kBlockN = 128;   // the only instantiation width (osvos_conv3x3_wgrad above)
  WgradParams p;
  int grid = 0;
  rc = plan_wgrad(a, kBlockN, device_sm_count(), wgrad_switches(), p, grid);
  if (rc) {
    set_last_error("osvos_conv3x3_wgrad_plan: dz_channels = %d cannot be tiled", a->dz_channels);
    return rc;
  }
  memset(plan, 0, sizeof(*plan));
  plan->block_n = kBlockN;
  plan->planes = fast ? 1 : 2;
  plan->split_acc = fast ? WgCfg<kBlockN, 1>::kSplitAcc : WgCfg<kBlockN, 2>::kSplitAcc;
  plan->lean = 0;
  plan->items = p.total_items;
  plan->grid = grid;
  plan->tap_mode = p.tap_rows ? OSVOS_TAP_ROWS : p.tap_pairs ? OSVOS_TAP_PAIRS : OSVOS_TAP_NINE;
  plan->pixel_splits = p.splits;
  return OSVOS_OK;
}
