// 3x3 convolution as a tcgen05 implicit GEMM with HALO REUSE (sm_100a).
//
// GEMM view: M = 128 output pixels (8 px x 16 rows), N = BLOCK_N output channels, K = 9 taps x Cin; split-bf16
// operands; warp 0 is the TMA producer, warp 1 the MMA issuer, the others run the epilogue (conv_common.cuh).
// The activation operand is loaded ONCE per (tile, 64-channel chunk) as the 18-row x 10-px halo patch and the nine taps
// are nine UMMA smem descriptors into it: tap (r, s) starts at smem row (r * PITCH + s); the 16 tile rows are the sixteen
// 8-row swizzle groups at stride SBO = PITCH * 128 B.  That divides the activation traffic through L2 -> smem by ~6
// relative to one shifted box per tap, which is what bounded the earlier per-tap kernel (DESIGN.md section 4).  The
// weight slabs stream through their own, deeper ring (one stage per tap), and the next chunk's halo is prefetched while
// the current one is being consumed.
//
// PITCH is the smem row pitch in pixels: 10 packs the patch rows (1280 B) and relies on the UMMA swizzle being a
// function of the absolute shared-memory address, validated on hardware together with the padded 16-pixel pitch and the
// descriptor's base-offset field in round 1 (the base-offset field must stay 0).
//
// Producer and issuer loops: one elected thread each, taps unrolled, descriptors by addition - see the comments at
// the two loops and DESIGN.md section 4 for the measurements behind that.
#include <string.h>

#include <type_traits>

#include "conv_common.cuh"

namespace osvos {

constexpr int kHaloRows = kTileH + 2;  // 18

template <int BLOCK_N, int PLANES, int PITCH, bool SPLIT, bool LEAN = false>
struct HaloCfg {
  static constexpr int kABoxBytes = kHaloRows * PITCH * 128;                // one plane, one chunk
  static constexpr int kAPlaneBytes = (kABoxBytes + 1023) / 1024 * 1024;    // keep 1 KiB alignment
  static constexpr int kAStageBytes = PLANES * kAPlaneBytes;
  static constexpr int kAStages = 2;
  static constexpr int kBPlaneBytes = BLOCK_N * 128;
  static constexpr int kBStageBytes = PLANES * kBPlaneBytes;
  // LEAN: the forward-only epilogue (conv_common.cuh: conv_epilogue_lean) instead of the general one.
  static constexpr int kBudget = 225 * 1024 - kAStages * kAStageBytes;   // 227 KiB per CTA minus align/barriers
  static constexpr int kBStagesRaw = kBudget / kBStageBytes;
  static constexpr int kBStages = kBStagesRaw > 9 ? 9 : kBStagesRaw;
  // Exact mode with BLOCK_N <= 128: N-concatenated split-B.  The hi and lo weight planes are contiguous in the B
  // stage, so ONE tcgen05.mma of N = 2 * BLOCK_N computes [A_hi.B_hi | A_hi.B_lo] into two column halves of the
  // accumulator; with the N = BLOCK_N pass A_lo.B_hi that is 2 instructions per K step instead of 3 (the per-
  // instruction floor of ~85 cycles makes instruction count, not flops, the cost).  The epilogue adds the halves.
  static constexpr bool kSplitAcc = SPLIT;
  static_assert(!SPLIT || (PLANES == 2 && BLOCK_N <= 128), "split accumulators need two planes and 2 * BLOCK_N <= 256");
  static constexpr int kAccCols = kSplitAcc ? 2 * BLOCK_N : BLOCK_N;
  static constexpr int kTmemCols = (2 * kAccCols) < 32 ? 32 : 2 * kAccCols;
  static constexpr int kSmemBytes = kAStages * kAStageBytes + kBStages * kBStageBytes + 1024 + 512;
  static_assert(kBStages >= 2, "weight ring too shallow");
  // The issuer forms descriptors by ADDING (bytes >> 4) to a base descriptor: every address it can reach - the end of
  // the dynamic allocation plus the static shared variables' 1 KiB alignment slack - must stay inside the 14-bit
  // start-address field (256 KiB), or the add would carry into the leading-dimension field.
  static_assert(kSmemBytes <= 227 * 1024, "more than the per-CTA shared memory of sm_100");
  static_assert(kSmemBytes + 4096 < (1 << 18), "descriptor start-address field would overflow");
  static_assert(kBStageBytes % 1024 == 0, "B stage must keep 1024-byte alignment");
};

template <int BLOCK_N, int PLANES, int PITCH, bool SPLIT, bool LEAN>
__global__ void __launch_bounds__(64 + EpiCfg<BLOCK_N>::kThreads, 1)
conv3x3_halo_kernel(const __grid_constant__ CUtensorMap map_x_hi, const __grid_constant__ CUtensorMap map_x_lo,
                    const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                    const ConvParams p) {
  using Cfg = HaloCfg<BLOCK_N, PLANES, PITCH, SPLIT, LEAN>;
  constexpr int SA = Cfg::kAStages, SB = Cfg::kBStages;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + SA * Cfg::kAStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + SB * Cfg::kBStageBytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + SA;
  uint64_t* b_full = bars + 2 * SA;
  uint64_t* b_empty = bars + 2 * SA + SB;
  uint64_t* tfull_bar = bars + 2 * SA + 2 * SB;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_x_hi);
    tma_prefetch_desc(&map_w_hi);
    if (PLANES == 2) {
      tma_prefetch_desc(&map_x_lo);
      tma_prefetch_desc(&map_w_lo);
    }
    for (int i = 0; i < SA; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < SB; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], EpiCfg<BLOCK_N>::kThreads);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above touched only shared memory, TMEM and the kernel parameters; the previous kernel's
  // outputs (activations, masks, pooled planes, workspaces) are first accessed below.
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (one elected thread)
    // Same economy as the MMA issuer below: ONE elected thread runs the whole loop (no per-step ELECT / warp
    // reconvergence), taps unrolled (the tap coordinate is an immediate), tile coordinates decoded once per tile
    // (three integer divisions) instead of once per halo load.
    if (elect_one()) {
      int a_stage = 0, b_stage = 0;
      uint32_t a_phase = 0, b_phase = 0;
      const bool skip_a = (p.ablate & 2) != 0, skip_b = (p.ablate & 1) != 0;
      auto issue_a = [&](int x0, int y0, int img, int kc) {
        mbar_wait(&a_empty[a_stage], a_phase ^ 1);
        if (skip_a) {
          mbar_arrive(&a_full[a_stage]);
        } else {
          uint8_t* st = smem_a + a_stage * Cfg::kAStageBytes;
          mbar_arrive_expect_tx(&a_full[a_stage], PLANES * Cfg::kABoxBytes);
          tma_load_4d(&map_x_hi, &a_full[a_stage], st, kc * kBlockK, x0, y0, img);
          if (PLANES == 2) tma_load_4d(&map_x_lo, &a_full[a_stage], st + Cfg::kAPlaneBytes, kc * kBlockK, x0, y0, img);
        }
        if (++a_stage == SA) {
          a_stage = 0;
          a_phase ^= 1;
        }
      };
      int nb = 0, tx = 0, ty = 0, img = 0;
      const int w_first = static_cast<int>(blockIdx.x), w_stride = static_cast<int>(gridDim.x);
      if (w_first < p.total_tiles) {
        decode_tile(p, w_first, nb, tx, ty, img);
        issue_a(tx * kTileW - 1, ty * kTileH - 1, img, 0);
      }
      for (int tile = w_first; tile < p.total_tiles; tile += w_stride) {
        const bool has_next = tile + w_stride < p.total_tiles;
        int nnb = 0, ntx = 0, nty = 0, nimg = 0;
        if (has_next) decode_tile(p, tile + w_stride, nnb, ntx, nty, nimg);
        const int n0 = nb * BLOCK_N;
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          const int c0 = kc * kBlockK;
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            if (tap == 3) {  // prefetch the next chunk's halo while this one is being consumed
              if (kc + 1 < p.k_chunks) issue_a(tx * kTileW - 1, ty * kTileH - 1, img, kc + 1);
              else if (has_next) issue_a(ntx * kTileW - 1, nty * kTileH - 1, nimg, 0);
            }
            mbar_wait(&b_empty[b_stage], b_phase ^ 1);
            if (skip_b) {
              mbar_arrive(&b_full[b_stage]);
            } else {
              uint8_t* st = smem_b + b_stage * Cfg::kBStageBytes;
              mbar_arrive_expect_tx(&b_full[b_stage], Cfg::kBStageBytes);
              tma_load_3d(&map_w_hi, &b_full[b_stage], st, c0, n0, tap);
              if (PLANES == 2) tma_load_3d(&map_w_lo, &b_full[b_stage], st + Cfg::kBPlaneBytes, c0, n0, tap);
            }
            if (++b_stage == SB) {
              b_stage = 0;
              b_phase ^= 1;
            }
          }
        }
        nb = nnb, tx = ntx, ty = nty, img = nimg;
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // -------------------------------------------------------------- MMA issuer (one elected thread)
    // The per-tap scalar work of this warp is what bounds the kernel, not the tensor pipe: timing ablations
    // (scripts/ablate.py, profiles/r01f_ablation_480p.txt) showed that with every load, MMA and store removed the
    // barrier skeleton alone still took 50-100 % of the full time, i.e. 600-900 cycles per (tap, 64-channel) step
    // against 448 (N = 64) / 768 (N = 128) cycles of MMA time, while a bare issue loop sustains 48 / 64 cycles per
    // MMA (scripts/microbench/operand_reuse_bench.cu).  So: the nine taps are unrolled (tap offsets are immediates),
    // descriptors are formed by ADDING to one per-chunk base instead of being rebuilt, and nothing is recomputed
    // per K step.  (A negative result from before, for the record: flattening the (tile, chunk, tap) nest to probe
    // the next step's barrier between MMAs was 8 % slower - more index math on this warp.)
    {
      constexpr uint32_t idesc = make_idesc_f16(kBlockM, BLOCK_N, /*bf16=*/true);
      constexpr uint32_t idesc2 = make_idesc_f16(kBlockM, Cfg::kSplitAcc ? 2 * BLOCK_N : BLOCK_N, /*bf16=*/true);
      // descriptor templates without the start-address field (bits [0,14) = address >> 4): adding (bytes >> 4) to a
      // descriptor moves its start address (shared-memory addresses stay below 2^18, no carry out of the field)
      constexpr uint64_t kDescA = (static_cast<uint64_t>(16 >> 4) << 16) | (static_cast<uint64_t>((PITCH * 128) >> 4) << 32) |
                                  (1ull << 46) | (static_cast<uint64_t>(kLayoutSW128) << 61);
      constexpr uint64_t kDescB = (static_cast<uint64_t>(16 >> 4) << 16) | (static_cast<uint64_t>(1024 >> 4) << 32) |
                                  (1ull << 46) | (static_cast<uint64_t>(kLayoutSW128) << 61);
      constexpr uint32_t kLoPlaneA = Cfg::kAPlaneBytes >> 4, kLoPlaneB = Cfg::kBPlaneBytes >> 4;
      const uint32_t smem_a_u32 = smem_u32(smem_a), smem_b_u32 = smem_u32(smem_b);
      const int k_steps = (p.ablate & 4) ? 0 : p.k_steps;   // < 4 only for zero-padded input channels (k_valid)
      // One tap = wait for its weight slab, FULLK ? 8 : up to 8 MMAs, release the slab.  FULLK (all four K steps of
      // the 64-channel chunk) is the common case and has no per-K-step branches.
      auto run = [&](auto fullk_tag) {
        constexpr bool FULLK = decltype(fullk_tag)::value;
        int a_stage = 0, b_stage = 0;
        uint32_t a_phase = 0, b_phase = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
          const int as = it & 1;
          const uint32_t aph = (it >> 1) & 1;
          mbar_wait(&tempty_bar[as], aph ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + as * Cfg::kAccCols;
          for (int kc = 0; kc < p.k_chunks; ++kc) {
            mbar_wait(&a_full[a_stage], a_phase);
            tc_fence_after();
            const uint64_t da0 = kDescA | static_cast<uint64_t>((smem_a_u32 + a_stage * Cfg::kAStageBytes) >> 4);
            const uint32_t not_first_chunk = kc != 0;
            const bool last_chunk = kc == p.k_chunks - 1;
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              constexpr int kRowBytes16 = 128 >> 4;
              const uint32_t tap_off = static_cast<uint32_t>(((tap / 3) * PITCH + (tap % 3)) * kRowBytes16);
              mbar_wait(&b_full[b_stage], b_phase);
              tc_fence_after();
              const uint64_t db_hi = kDescB | static_cast<uint64_t>((smem_b_u32 + b_stage * Cfg::kBStageBytes) >> 4);
              {
                const uint64_t da_hi = da0 + tap_off;
                const uint64_t da_lo = da_hi + kLoPlaneA;
#pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k) {
                  if (FULLK || k < k_steps) {
                    const uint32_t acc = (tap == 0 && k == 0) ? not_first_chunk : 1u;
                    if (Cfg::kSplitAcc) {
                      umma_f16(tmem_d, da_hi + 2 * k, db_hi + 2 * k, idesc2, acc);   // [A_hi.B_hi | A_hi.B_lo], N = 2 * BLOCK_N
                      umma_f16(tmem_d, da_lo + 2 * k, db_hi + 2 * k, idesc, 1);      // + A_lo.B_hi into the first half
                    } else if (PLANES == 2) {
                      umma_f16(tmem_d, da_lo + 2 * k, db_hi + 2 * k, idesc, acc);
                      umma_f16(tmem_d, da_hi + 2 * k, db_hi + kLoPlaneB + 2 * k, idesc, 1);
                      umma_f16(tmem_d, da_hi + 2 * k, db_hi + 2 * k, idesc, 1);
                    } else {
                      umma_f16(tmem_d, da_hi + 2 * k, db_hi + 2 * k, idesc, acc);
                    }
                  }
                }
                umma_commit(&b_empty[b_stage]);
                if (tap == 8) {
                  umma_commit(&a_empty[a_stage]);
                  if (last_chunk) umma_commit(&tfull_bar[as]);
                }
              }
              if (++b_stage == SB) {
                b_stage = 0;
                b_phase ^= 1;
              }
            }
            if (++a_stage == SA) {
              a_stage = 0;
              a_phase ^= 1;
            }
          }
        }
      };
      // ONE elected thread runs the whole issue loop (waits included): no per-tap ELECT / BSSY / BSYNC / warp
      // reconvergence; the other 31 lanes go straight to the closing __syncthreads.
      if (elect_one()) {
        if (k_steps == kBlockK / 16) run(std::true_type{});
        else run(std::false_type{});
      }
      __syncwarp();
    }
  } else {
    if constexpr (LEAN) conv_epilogue_lean<BLOCK_N>(p, tmem_base, tfull_bar, tempty_bar, warp, lane);
    else conv_epilogue_loop<BLOCK_N, Cfg::kSplitAcc>(p, tmem_base, tfull_bar, tempty_bar, warp, lane);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// The dispatcher's switches: OSVOS_HALO_LEAN, OSVOS_CONV_N256, OSVOS_SPLITACC128 (runtime.cu).
struct HaloSwitches {
  bool lean, n256, splitacc128;
};
static HaloSwitches halo_switches() {
  return HaloSwitches{env_int("OSVOS_HALO_LEAN", 1) != 0, env_int("OSVOS_CONV_N256", 1) != 0,
                      env_int("OSVOS_SPLITACC128", 1) != 0};
}

template <int BLOCK_N, int PLANES, int PITCH, bool SPLIT = (PLANES == 2 && BLOCK_N <= 128), bool LEAN = false>
static int launch_halo(const osvos_conv3x3_args* a, cudaStream_t stream) {
  using Cfg = HaloCfg<BLOCK_N, PLANES, PITCH, SPLIT, LEAN>;
  ConvParams p;
  fill_conv_params(p, a, BLOCK_N);
  CUtensorMap mx_hi, mx_lo, mw_hi, mw_lo;
  int rc = encode_act_maps(&mx_hi, &mx_lo, a->x_hi, PLANES == 2 ? a->x_lo : nullptr, a->n, a->h, a->w, a->cin, PITCH,
                           kHaloRows);
  if (rc) return rc;
  rc = encode_weight_maps(&mw_hi, &mw_lo, a->w_packed, a->cout, a->cin, BLOCK_N, 1);
  if (rc) return rc;
  OSVOS_CHECK_CUDA((launch_persistent<conv3x3_halo_kernel<BLOCK_N, PLANES, PITCH, SPLIT, LEAN>>(
      p.total_tiles, 64 + EpiCfg<BLOCK_N>::kThreads, Cfg::kSmemBytes, stream, mx_hi, mx_lo, mw_hi, mw_lo, p)));
  return OSVOS_OK;
}

// What dispatch_halo launches: the instantiation and the persistent grid.  One pure function of the arguments, the SM
// count and the switches, so that osvos_conv3x3_plan reports exactly what osvos_conv3x3 runs.
struct HaloChoice {
  int block_n, planes;
  bool split, lean;
};
static HaloChoice choose_halo(const osvos_conv3x3_args* a, int sms, const HaloSwitches& sw) {
  const bool fast = (a->flags & OSVOS_FLAG_FAST) != 0;
  if (a->cout == 16) return fast ? HaloChoice{16, 1, false, false} : HaloChoice{16, 2, true, false};
  // the lean epilogue serves launches that use nothing but bias / ReLU / split-bf16 act output / fused pool (exact mode)
  const bool lean = sw.lean && !fast && !(a->flags & OSVOS_FLAG_RELU_MASK) && a->colsum == nullptr && a->y_f32 == nullptr &&
                    a->pq == nullptr && (a->y_hi != nullptr || a->pool_hi != nullptr) &&
                    (a->y_hi == nullptr || a->y_lo != nullptr) && (a->pool_hi == nullptr || a->pool_lo != nullptr) &&
                    a->k_valid == 0;
  const HaloChoice n64 = lean ? HaloChoice{64, 2, true, true} : fast ? HaloChoice{64, 1, false, false} : HaloChoice{64, 2, true, false};
  if (a->cout == 64) return n64;
  const int m_tiles = ((a->w + kTileW - 1) / kTileW) * ((a->h + kTileH - 1) / kTileH) * a->n;
  const long tiles128 = static_cast<long>(m_tiles) * (a->cout / 128);
  const long waves128 = (tiles128 + sms - 1) / sms;
  const long waves256 = (static_cast<long>(m_tiles) * (a->cout / 256) + sms - 1) / sms;
  // few tiles (stage 5 at 480x854: 56 of 128 x 128): N = 64 tiles double the CTA count at ~0.8x the time per tile.
  // (Stream-K - (tile, chunk) units in balanced contiguous ranges, tiles cut by a range boundary exchanging fp32 partial
  // accumulators - was built, validated and measured in round 2: -18 % on 240x427 frames and -5 % at 480x854 when
  // applied to every badly quantised layer, -1 % / +-0 / +2 % (240p / 480p / 720p) when restricted to layers with at
  // least one whole tile per CTA.  The layers it would help are power-limited: the idle SMs of a ragged last wave are
  // what lets the busy ones clock higher.  Removed again; profiles/r02c_ab_matrix.txt, r02d_ab_matrix_*.txt.)
  if (waves128 == 1 && tiles128 * 5 <= static_cast<long>(sms) * 3) return n64;
  // N = 256 tiles (one tcgen05.mma of 128 cycles per pass) whenever that does not cost a wave; measured cycles per
  // (tap, 64-channel) step: N = 128 ~ 1000 (2 + 1 instructions), N = 256 ~ 2200 exact.  (Exact mode never prefers
  // them: waves128 <= 2 * waves256 whenever cout % 256 == 0.)
  const bool prefer256 = fast ? waves256 * 1100 < waves128 * 700 : waves256 * 2200 < waves128 * 1000;
  if (a->cout % 256 == 0 && prefer256 && sw.n256) return fast ? HaloChoice{256, 1, false, false} : HaloChoice{256, 2, false, false};
  if (fast) return HaloChoice{128, 1, false, false};
  // Exact mode, N = 128: the N-concatenated split accumulator (2 MMAs per K step, 256 accumulator columns, the
  // epilogue sums two halves) and the plain three-pass form (3 MMAs, 128 columns) cost the SAME tensor time
  // (scripts/microbench/operand_reuse_bench.cu) and measured the same; OSVOS_SPLITACC128=0 selects the three-pass form.
  if (!sw.splitacc128) return HaloChoice{128, 2, false, false};
  return HaloChoice{128, 2, true, lean};
}

template <int PITCH>
static int dispatch_halo(const osvos_conv3x3_args* a, cudaStream_t stream) {
  const HaloChoice c = choose_halo(a, device_sm_count(), halo_switches());
#define OSVOS_HALO_CASE(BN, PL, SP, LE) \
  if (c.block_n == BN && c.planes == PL && c.split == SP && c.lean == LE) return launch_halo<BN, PL, PITCH, SP, LE>(a, stream)
  OSVOS_HALO_CASE(16, 1, false, false);
  OSVOS_HALO_CASE(16, 2, true, false);
  OSVOS_HALO_CASE(64, 1, false, false);
  OSVOS_HALO_CASE(64, 2, true, false);
  OSVOS_HALO_CASE(64, 2, true, true);
  OSVOS_HALO_CASE(128, 1, false, false);
  OSVOS_HALO_CASE(128, 2, false, false);
  OSVOS_HALO_CASE(128, 2, true, false);
  OSVOS_HALO_CASE(128, 2, true, true);
  OSVOS_HALO_CASE(256, 1, false, false);
  OSVOS_HALO_CASE(256, 2, false, false);
#undef OSVOS_HALO_CASE
  set_last_error("conv3x3: no halo instantiation for N = %d, %d plane(s), split %d, lean %d", c.block_n, c.planes,
                 (int)c.split, (int)c.lean);
  return OSVOS_ERR_UNSUPPORTED;
}

int conv3x3_halo_dispatch(const osvos_conv3x3_args* a, cudaStream_t stream) {
  // packed patch rows (pitch 10) are the only instantiation: the padded 16-pixel pitch and the descriptor base-offset
  // field were validated equivalent on hardware in round 1 and dropped
  return dispatch_halo<10>(a, stream);
}

static int check_conv_args(const osvos_conv3x3_args* a) {
  OSVOS_CHECK_ARG(a != nullptr);
  OSVOS_CHECK_ARG(a->n > 0 && a->h > 0 && a->w > 0);
  OSVOS_CHECK_ARG(a->cin >= 64 && a->cin % 64 == 0);
  OSVOS_CHECK_ARG(a->cout == 2 || a->cout == 16 || a->cout == 64 || (a->cout > 0 && a->cout % 128 == 0));
  // cout == 2: the folded side branch (osvos_fold_side_weights) - pq is the only output, bias = the 2 folded biases
  OSVOS_CHECK_ARG(a->cout != 2 || (a->pq != nullptr && a->y_hi == nullptr && a->y_f32 == nullptr && a->pool_hi == nullptr &&
                                   a->colsum == nullptr && !(a->flags & (OSVOS_FLAG_RELU | OSVOS_FLAG_RELU_MASK)) &&
                                   a->k_valid == 0));
  OSVOS_CHECK_ARG(a->x_hi != nullptr && a->w_packed != nullptr);
  OSVOS_CHECK_ARG((a->flags & OSVOS_FLAG_FAST) || a->x_lo != nullptr);
  OSVOS_CHECK_ARG(a->y_hi != nullptr || a->y_f32 != nullptr || a->pq != nullptr || a->pool_hi != nullptr);
  OSVOS_CHECK_ARG(!(a->flags & OSVOS_FLAG_RELU_MASK) || a->mask_hi != nullptr);
  OSVOS_CHECK_ARG(a->pq == nullptr || a->cout == 2 || (a->cout == 16 && a->proj_w != nullptr));
  OSVOS_CHECK_ARG((a->pool_hi == nullptr && a->colsum == nullptr) || a->cout >= 64);
  OSVOS_CHECK_ARG((reinterpret_cast<uintptr_t>(a->x_hi) & 15) == 0);
  OSVOS_CHECK_ARG((reinterpret_cast<uintptr_t>(a->w_packed) & 15) == 0);
  OSVOS_CHECK_ARG((reinterpret_cast<uintptr_t>(a->bias) & 15) == 0);
  if (a->cout >= 64) {   // 256-bit stores / loads in the epilogues
    const uintptr_t any = reinterpret_cast<uintptr_t>(a->y_hi) | reinterpret_cast<uintptr_t>(a->y_lo) |
                          reinterpret_cast<uintptr_t>(a->y_f32) | reinterpret_cast<uintptr_t>(a->pool_hi) |
                          reinterpret_cast<uintptr_t>(a->pool_lo) | reinterpret_cast<uintptr_t>(a->mask_hi);
    OSVOS_CHECK_ARG((any & 31) == 0);
  }
  OSVOS_CHECK_ARG(a->k_valid >= 0 && a->k_valid <= 64 && a->k_valid % 16 == 0);
  return OSVOS_OK;
}

}  // namespace osvos

using namespace osvos;

extern "C" int osvos_side_folded_multi(const osvos_conv3x3_args* args, int count, osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(args != nullptr && count > 0 && count <= 4);
  const osvos_conv3x3_args* order[4];
  for (int k = 0; k < count; ++k) {
    int rc = check_conv_args(&args[k]);
    if (rc) return rc;
    OSVOS_CHECK_ARG(args[k].cout == 2);
    OSVOS_CHECK_ARG((args[k].flags & OSVOS_FLAG_FAST) == (args[0].flags & OSVOS_FLAG_FAST));
    order[k] = &args[k];
  }
  // deepest scale first: its tiles hold the most channel chunks, and the round-robin deal balances better that way
  for (int i = 1; i < count; ++i)
    for (int j = i; j > 0 && order[j]->cin > order[j - 1]->cin; --j) {
      const osvos_conv3x3_args* t = order[j];
      order[j] = order[j - 1];
      order[j - 1] = t;
    }
  return side_conv_multi_dispatch(order, count, static_cast<cudaStream_t>(stream_));
}

// side_prep shape (16 outputs, fp32 features / projections only): nine-taps-along-N kernel (side_conv.cu);
// OSVOS_SIDE_IMPL=generic sends it through the halo kernel's N = 16 instantiation instead (cross-check)
static bool routes_to_side_conv(const osvos_conv3x3_args* a) {
  if (a->cout == 2) return true;
  return a->cout == 16 && a->y_hi == nullptr && !(a->flags & OSVOS_FLAG_RELU_MASK) && a->colsum == nullptr &&
         !env_is("OSVOS_SIDE_IMPL", "generic");
}

extern "C" int osvos_conv3x3(const osvos_conv3x3_args* a, osvos_stream_t stream_) {
  int rc = check_conv_args(a);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (routes_to_side_conv(a)) return side_conv_dispatch(a, stream);
  return conv3x3_halo_dispatch(a, stream);
}

extern "C" int osvos_conv3x3_plan(const osvos_conv3x3_args* a, osvos_launch_plan* plan) {
  int rc = check_conv_args(a);
  if (rc) return rc;
  OSVOS_CHECK_ARG(plan != nullptr);
  if (routes_to_side_conv(a)) {
    set_last_error("osvos_conv3x3_plan: these arguments go to the side-branch kernel (side_conv.cu), not the halo kernel");
    return OSVOS_ERR_UNSUPPORTED;
  }
  const int sms = device_sm_count();
  const HaloChoice c = choose_halo(a, sms, halo_switches());
  memset(plan, 0, sizeof(*plan));
  plan->block_n = c.block_n;
  plan->planes = c.planes;
  plan->split_acc = c.split ? 1 : 0;
  plan->lean = c.lean ? 1 : 0;
  ConvParams p;
  fill_conv_params(p, a, c.block_n);
  plan->items = p.total_tiles;
  plan->grid = persistent_grid(p.total_tiles, sms);
  return OSVOS_OK;
}
