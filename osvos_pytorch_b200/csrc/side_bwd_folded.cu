// Backward of the side branch in FOLDED (rank-2) form - training path.
//
// side_prep[i] has no ReLU (reference networks/vgg_osvos.py:67), so the whole side branch of a scale,
//   feat = side_prep(x);  p = score_dsn(feat);  q = fuse_slice . feat            (:41,44,54 run at :67,69,72)
// is ONE linear 3x3 convolution C -> 2 with weights W'[o][c][t] = sum_f proj[o][f] * W_side[f][c][t] (the inference
// path already runs it that way, osvos_fold_side_weights).  Its backward therefore only ever sees the TWO gradient
// channels dpq = (dL/dp, dL/dq) - not the 16 feature gradients autograd materialises:
//
//   G[t][o][c] = sum_px dpq[px - t][o] * x[px][c]        "folded weight gradient": 18 numbers per channel     (1)
//   S[o]       = sum_px dpq[px][o]
//   dX[px][c]  = sum_{t,o} W'[o][c][t] * dpq[px - t][o]   gradient w.r.t. the stage output (before its ReLU)   (2)
//
// and every parameter gradient of the branch is algebra on G and S (side_grads_finish_kernel):
//   d side_prep.weight[f][c][t] = proj[0][f] G[t][0][c] + proj[1][f] G[t][1][c]
//   d side_prep.bias[f]         = proj[0][f] S[0]       + proj[1][f] S[1]
//   d score_dsn.weight[f]       = <W_side[f], G[.][0][.]> + b_side[f] S[0],     d score_dsn.bias = S[0]
//   d fuse.weight[16 i + f]     = <W_side[f], G[.][1][.]> + b_side[f] S[1]
// (1) reads the stage output ONCE on CUDA cores (18 FMAs per element, fp32 accumulate over hi + lo) instead of nine
// shifted passes of a 64-wide tensor-core wgrad whose N is 3/4 zero padding; (2) is 18 FMAs per element inside the
// max-unpool / ReLU-mask kernel that consumes it (bwd_kernels.cu), instead of a 3x3 dgrad convolution 16 -> C that
// wrote an fp32 map of the stage's size only to be read back once.  The 16 side features, their gradient and the padded
// 64-channel operand copies are never formed.  Replaces the autograd of networks/vgg_osvos.py:67,69,72 triggered at
// train_online.py:141 / train_parent.py:164.
#include "common.cuh"
#include "ptx.cuh"

namespace osvos {

constexpr int kSwSlab = 128;

// G[t][o][c] (+ S[2] behind it), t = 3 r + s.
// Work item = a CHUNK of 28 consecutive pixels of one image row x one 128-channel slab.  A block (seven compute warps + one
// producer warp; two blocks per SM) owns one slab (blockIdx % slabs) and walks the chunks of that slab round-robin, so that neighbouring
// blocks read neighbouring 7 KiB pieces of the map.  The producer warp streams the chunks through a four-stage ring: the
// 28 x 128-channel tile of each bf16 plane by ONE 2-D TMA box (the map is a [pixels, C] matrix), the 3 x 30 window of
// dpq by 8-byte cp.async copies that arrive on the same barrier.  Compute warp w takes pixels 4w .. 4w+3 of the chunk: its lane holds four
// channels x 18 accumulators; per pixel it reads 8 + 8 bytes of x and nine float2 of the window from shared memory.
// (History, stage-2 map of 52 MB at 480p: per-warp row segments with register prefetch, a dpq column and one pixel
// loaded per iteration: 54 us; window in shared memory + the next four pixels in flight: 44 us - 4,700 concurrent
// 256-byte streams kept DRAM at 1.3 TB/s with 2.5 us of load latency (profiles/r02l_ncu_side_folded_wgrad_v2.txt).)
constexpr int kSwChunk = 28;                       // pixels per chunk: four per compute warp
constexpr int kSwStages = 4;
constexpr int kSwTileBytes = kSwChunk * kSwSlab * 2;          // one plane: 8 KiB
constexpr int kSwWinBytes = 1024;                  // 3 x 30 float2 = 720 B
constexpr int kSwStageBytes = 2 * kSwTileBytes + kSwWinBytes;
static_assert(kSwTileBytes % 128 == 0 && kSwStageBytes % 128 == 0, "TMA destinations stay 128-byte aligned");
constexpr int kSwComputeWarps = 7;                  // + 1 producer warp = 256 threads: 128 registers at two blocks per SM
constexpr int kSwKernelThreads = (kSwComputeWarps + 1) * 32;
constexpr int kSwWinPerLane = (3 * (kSwChunk + 2) + 31) / 32;
static_assert(kSwComputeWarps * 4 == kSwChunk, "four pixels of a chunk per compute warp");
static_assert(3 * (kSwChunk + 2) * 8 <= kSwWinBytes, "window area");
constexpr int kSwPartBytes = kSwComputeWarps * 18 * kSwSlab * 4;            // 63 KiB of partial sums at the end
constexpr int kSwRingBytes = kSwStages * kSwStageBytes;
constexpr int kSwDataBytes = kSwPartBytes > kSwRingBytes ? kSwPartBytes : kSwRingBytes;
constexpr int kSwSmemBytes = kSwDataBytes + (2 * kSwComputeWarps + 2) * 4 + 2 * kSwStages * 8 + 128;
static_assert(kSwDataBytes % 8 == 0 && ((2 * kSwComputeWarps + 2) * 4) % 8 == 0, "mbarrier alignment");

// Up to four SCALES per launch (the backward runs the four side branches' G kernels as one): the grid is cut into one
// block range per scale, sized by the scale's chunk count, so the fixed cost of a launch (first tile's latency, block
// reduction, atomics: ~9 us of a 10 us launch on the 30 x 54 map) is paid once.
constexpr int kSwMaxScales = 4;
struct SwScale {
  const float* dpq;
  float* g;
  int n, h, w, c;
  int block_begin, blocks;       // this scale's blocks: [block_begin, block_begin + blocks), a multiple of c / 128
};
struct SwParams {
  SwScale sc[kSwMaxScales];
  int count;
  int has_lo;
};
struct SwMaps {
  CUtensorMap hi[kSwMaxScales], lo[kSwMaxScales];
};

__global__ void __launch_bounds__(kSwKernelThreads, 2)
side_folded_wgrad_kernel(const __grid_constant__ SwMaps maps, const __grid_constant__ SwParams p) {
  int sci = 0;
  while (sci + 1 < p.count && static_cast<int>(blockIdx.x) >= p.sc[sci + 1].block_begin) ++sci;
  const SwScale& L = p.sc[sci];
  const CUtensorMap& map_hi = maps.hi[sci];
  const CUtensorMap& map_lo = maps.lo[sci];
  const float* __restrict__ dpq = L.dpq;
  float* __restrict__ g = L.g;
  const int n = L.n, h = L.h, w = L.w, c = L.c, has_lo = p.has_lo;
  extern __shared__ uint8_t sw_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(sw_smem_raw) + 127) & ~uintptr_t(127));
  // after the last chunk the ring (+ the slack behind it) is reused for the warps' partial sums: [warp][18][128] floats
  float* part = reinterpret_cast<float*>(smem);
  float* part_s = reinterpret_cast<float*>(smem + kSwPartBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(part_s + 2 * kSwComputeWarps + 2);
  uint64_t* empty_bar = full_bar + kSwStages;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slabs = c / kSwSlab;
  const int lb = static_cast<int>(blockIdx.x) - L.block_begin;      // block index inside the scale's range
  const int slab = lb % slabs;
  const int blk = lb / slabs, nblk = L.blocks / slabs;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_hi);
    if (has_lo) tma_prefetch_desc(&map_lo);
    for (int i = 0; i < kSwStages; ++i) {
      mbar_init(&full_bar[i], 1 + 32);          // the TMA transaction + the 32 producer lanes' window copies
      mbar_init(&empty_bar[i], kSwComputeWarps);
    }
    fence_barrier_init();
  }
  __syncthreads();
  pdl_wait();               // dpq / x are outputs of earlier kernels of the stream (ptx.cuh)
  pdl_launch_dependents();

  const int cpr = (w + kSwChunk - 1) / kSwChunk;                 // chunks per image row
  const int chunks = n * h * cpr;

  if (warp == kSwComputeWarps) {
    // ------------------------------------------------------------------ producer warp
    // Per chunk and stage: the 3 x 30 window of dpq by 8-byte cp.async with zero fill outside the image (window entry
    // idx = r * 30 + k <-> dpq[(y + 1 - r, x0 - 1 + k)]; up to kSwWinPerLane entries per lane), each lane's copies arriving
    // on the stage's full barrier when they land, and the two x tiles by TMA - nothing here waits for memory, so all four
    // stages are in flight.  (With the window prefetched ONE chunk ahead into registers the producer handed over one chunk
    // per load latency: 34 us for the stage-2 map.)
    int stage = 0;
    uint32_t phase = 0;
    for (int ci = blk; ci < chunks; ci += nblk) {
      const int cx = ci % cpr, row = ci / cpr;
      const int y = row % h, img = row / h, x0 = cx * kSwChunk;
      mbar_wait(&empty_bar[stage], phase ^ 1);
      uint8_t* st = smem + stage * kSwStageBytes;
      float2* win = reinterpret_cast<float2*>(st + 2 * kSwTileBytes);
#pragma unroll
      for (int j = 0; j < kSwWinPerLane; ++j) {
        const int idx = lane + 32 * j;
        if (idx < 3 * (kSwChunk + 2)) {
          const int r = idx / (kSwChunk + 2), k = idx - r * (kSwChunk + 2);
          const int yy = y + 1 - r, xx = x0 - 1 + k;
          const bool in = yy >= 0 && yy < h && xx >= 0 && xx < w;
          const float2* src = reinterpret_cast<const float2*>(dpq) + (in ? (static_cast<size_t>(img) * h + yy) * w + xx : 0);
          cp_async_8_zfill(win + idx, src, in ? 8u : 0u);
        }
      }
      cp_async_mbar_arrive_noinc(&full_bar[stage]);
      if (lane == 0) {
        const int pix0 = row * w + x0;                                // flat pixel index of the chunk's first pixel
        mbar_arrive_expect_tx(&full_bar[stage], (has_lo ? 2 : 1) * kSwTileBytes);
        tma_load_2d(&map_hi, &full_bar[stage], st, slab * kSwSlab, pix0);
        if (has_lo) tma_load_2d(&map_lo, &full_bar[stage], st + kSwTileBytes, slab * kSwSlab, pix0);
      }
      if (++stage == kSwStages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------------ compute warps
    float acc[9][2][4];
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int o = 0; o < 2; ++o)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[t][o][j] = 0.f;
    float s0 = 0.f, s1 = 0.f;
    int stage = 0;
    uint32_t phase = 0;
    for (int ci = blk; ci < chunks; ci += nblk) {
      const int cx = ci % cpr;
      const int valid = min(kSwChunk, w - cx * kSwChunk);            // pixels of this chunk inside the row
      mbar_wait(&full_bar[stage], phase);
      const uint8_t* st = smem + stage * kSwStageBytes;
      const float2* win = reinterpret_cast<const float2*>(st + 2 * kSwTileBytes);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int px = warp * 4 + u;
        if (px < valid) {
          const uint2 rh = *reinterpret_cast<const uint2*>(st + px * (kSwSlab * 2) + lane * 8);
          uint2 rl = make_uint2(0, 0);
          if (has_lo) rl = *reinterpret_cast<const uint2*>(st + kSwTileBytes + px * (kSwSlab * 2) + lane * 8);
          float v[4];
          v[0] = bf16_lo_to_float(rh.x) + bf16_lo_to_float(rl.x);
          v[1] = bf16_hi_to_float(rh.x) + bf16_hi_to_float(rl.x);
          v[2] = bf16_lo_to_float(rh.y) + bf16_lo_to_float(rl.y);
          v[3] = bf16_hi_to_float(rh.y) + bf16_hi_to_float(rl.y);
#pragma unroll
          for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int s = 0; s < 3; ++s) {
              const float2 d = win[r * (kSwChunk + 2) + px + 2 - s];       // dpq[px - t], t = (r - 1, s - 1)
              if (r == 1 && s == 1) {
                s0 += d.x;
                s1 += d.y;
              }
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                acc[3 * r + s][0][j] = fmaf(d.x, v[j], acc[3 * r + s][0][j]);
                acc[3 * r + s][1][j] = fmaf(d.y, v[j], acc[3 * r + s][1][j]);
              }
            }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[stage]);
      if (++stage == kSwStages) {
        stage = 0;
        phase ^= 1;
      }
    }
    // every compute warp is through with the ring: its memory now holds the warps' partial sums (see below)
    asm volatile("bar.sync 1, %0;" ::"n"(kSwComputeWarps * 32) : "memory");
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int o = 0; o < 2; ++o)
        *reinterpret_cast<float4*>(part + (warp * 18 + 2 * t + o) * kSwSlab + lane * 4) =
            make_float4(acc[t][o][0], acc[t][o][1], acc[t][o][2], acc[t][o][3]);
    if (lane == 0) {   // every lane of a warp saw the same dpq: one lane counts
      part_s[2 * warp] = s0;
      part_s[2 * warp + 1] = s1;
    }
  }
  __syncthreads();
  // Block reduction over the seven warps' partials (plain loads in a fixed order - the float atomicAdd on shared memory the
  // first versions used is a compare-and-swap loop, 72 of them per thread under 7-way contention), then one vector atomic
  // per (tap, o, 4 channels) and block.
  for (int i = threadIdx.x; i < 18 * (kSwSlab / 4); i += kSwKernelThreads) {
    float4 val = *reinterpret_cast<const float4*>(part + i * 4);
#pragma unroll
    for (int wv = 1; wv < kSwComputeWarps; ++wv) {
      const float4 v = *reinterpret_cast<const float4*>(part + wv * 18 * kSwSlab + i * 4);
      val.x += v.x, val.y += v.y, val.z += v.z, val.w += v.w;
    }
    const int to = i / (kSwSlab / 4), c4 = i % (kSwSlab / 4);
    atomicAdd(reinterpret_cast<float4*>(g + static_cast<size_t>(to) * c + slab * kSwSlab + c4 * 4), val);
  }
  if (slab == 0 && threadIdx.x < 2) {
    float v = 0.f;
#pragma unroll
    for (int wv = 0; wv < kSwComputeWarps; ++wv) v += part_s[2 * wv + threadIdx.x];
    atomicAdd(g + static_cast<size_t>(18) * c + threadIdx.x, v);
  }
}

// Parameter gradients of the side branch of up to four scales from G / S: one block per (scale, feature f).
struct SideGradScale {
  const float* g;        // [18][c] + S[2]
  const float* side_w;   // [16][c][9]
  const float* side_b;   // [16] or null
  const float* proj;     // [32]
  float* d_side_w;       // [16][c][9]
  float* d_side_b;       // [16]
  float* d_score_w;      // [16] or null
  float* d_score_b;      // [1] or null
  float* d_fuse_w;       // [16] or null
  int c;
  int accumulate;
};
struct SideGradTable {
  SideGradScale s[4];
  int count;
};

constexpr int kFinThreads = 1024;
__global__ void __launch_bounds__(kFinThreads) side_grads_finish_kernel(const __grid_constant__ SideGradTable t) {
  extern __shared__ float gs[];            // G of this block's scale: 18 rows of c floats at pitch c + 1 (bank spread), S[2]
  const SideGradScale& L = t.s[blockIdx.x / 16];
  const int f = blockIdx.x % 16;
  const int c = L.c, pitch = c + 1;
  pdl_wait();
  pdl_launch_dependents();
  for (int i = threadIdx.x; i < 18 * c; i += kFinThreads) gs[(i / c) * pitch + i % c] = __ldcg(L.g + i);
  if (threadIdx.x < 2) gs[18 * pitch + threadIdx.x] = __ldcg(L.g + 18 * c + threadIdx.x);
  __syncthreads();
  const float ps = __ldg(L.proj + f), pf = __ldg(L.proj + 16 + f);
  const float S0 = gs[18 * pitch], S1 = gs[18 * pitch + 1];
  float dot0 = 0.f, dot1 = 0.f;
  const float* __restrict__ wrow = L.side_w + static_cast<size_t>(f) * c * 9;
  float* __restrict__ drow = L.d_side_w + static_cast<size_t>(f) * c * 9;
  const bool accumulate = L.accumulate != 0;
#pragma unroll 2
  for (int i = threadIdx.x; i < c * 9; i += kFinThreads) {
    const int ci = i / 9, tap = i - ci * 9;
    const float g0 = gs[2 * tap * pitch + ci];
    const float g1 = gs[(2 * tap + 1) * pitch + ci];
    const float wv = __ldg(wrow + i);
    dot0 = fmaf(wv, g0, dot0);
    dot1 = fmaf(wv, g1, dot1);
    const float dv = fmaf(ps, g0, pf * g1);
    drow[i] = accumulate ? drow[i] + dv : dv;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    dot0 += __shfl_xor_sync(0xffffffffu, dot0, off);
    dot1 += __shfl_xor_sync(0xffffffffu, dot1, off);
  }
  __shared__ float r0[kFinThreads / 32], r1[kFinThreads / 32];
  if ((threadIdx.x & 31) == 0) {
    r0[threadIdx.x >> 5] = dot0;
    r1[threadIdx.x >> 5] = dot1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int i = 0; i < kFinThreads / 32; ++i) {
      a += r0[i];
      b += r1[i];
    }
    const float bs = L.side_b ? __ldg(L.side_b + f) : 0.f;
    auto put = [&](float* dst, float v) {
      if (dst) *dst = accumulate ? *dst + v : v;
    };
    put(L.d_side_b + f, fmaf(ps, S0, pf * S1));
    if (L.d_score_w) put(L.d_score_w + f, fmaf(bs, S0, a));
    if (L.d_fuse_w) put(L.d_fuse_w + f, fmaf(bs, S1, b));
    if (L.d_score_b && f == 0) put(L.d_score_b, S0);
  }
}

}  // namespace osvos

using namespace osvos;

extern "C" size_t osvos_side_folded_wgrad_floats(int c) { return static_cast<size_t>(18) * c + 2; }

extern "C" int osvos_side_folded_wgrad_multi(const osvos_side_wgrad_item* items, int count, osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(items != nullptr && count > 0 && count <= kSwMaxScales);
  SwParams p;
  SwMaps maps;
  memset(&p, 0, sizeof(p));
  p.count = count;
  p.has_lo = items[0].x_lo != nullptr ? 1 : 0;
  long work[kSwMaxScales], total_work = 0;
  for (int k = 0; k < count; ++k) {
    const osvos_side_wgrad_item& it = items[k];
    OSVOS_CHECK_ARG(it.x_hi != nullptr && it.dpq != nullptr && it.g != nullptr && it.n > 0 && it.h > 0 && it.w > 0);
    OSVOS_CHECK_ARG(it.c >= kSwSlab && it.c % kSwSlab == 0);
    OSVOS_CHECK_ARG((it.x_lo != nullptr) == (p.has_lo != 0));
    OSVOS_CHECK_ARG((reinterpret_cast<uintptr_t>(it.g) & 15) == 0 && (reinterpret_cast<uintptr_t>(it.x_hi) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(it.x_lo) & 15) == 0);
    const long npix = static_cast<long>(it.n) * it.h * it.w;
    const long chunks = static_cast<long>(it.n) * it.h * ((it.w + kSwChunk - 1) / kSwChunk);
    OSVOS_CHECK_ARG(npix < (1l << 31) && chunks < (1l << 30));
    SwScale& L = p.sc[k];
    L.dpq = it.dpq;
    L.g = it.g;
    L.n = it.n;
    L.h = it.h;
    L.w = it.w;
    L.c = it.c;
    work[k] = chunks * (it.c / kSwSlab);
    total_work += work[k];
    const uint64_t dims[2] = {(uint64_t)it.c, (uint64_t)npix};
    const uint64_t strides[1] = {(uint64_t)it.c * 2};
    const uint32_t box[2] = {kSwSlab, kSwChunk};
    int rc = encode_tensor_map(&maps.hi[k], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 2, it.x_hi, dims, strides, box,
                               CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    rc = encode_tensor_map(&maps.lo[k], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 2, it.x_lo ? it.x_lo : it.x_hi, dims, strides,
                           box, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
  }
  for (int k = count; k < kSwMaxScales; ++k) {   // unused slots: valid descriptors (never dereferenced)
    maps.hi[k] = maps.hi[0];
    maps.lo[k] = maps.lo[0];
  }
  // blocks per scale: its share of two blocks per SM by chunk count, a multiple of its slab count, at least one block per
  // slab and at most one block per chunk
  const long budget = static_cast<long>(device_sm_count()) * 2;
  int begin = 0;
  for (int k = 0; k < count; ++k) {
    const int slabs = p.sc[k].c / kSwSlab;
    const long chunks = work[k] / slabs;
    long b = (budget * work[k] + total_work / 2) / total_work / slabs;
    if (b < 1) b = 1;
    if (b > chunks) b = chunks;
    p.sc[k].block_begin = begin;
    p.sc[k].blocks = static_cast<int>(b * slabs);
    begin += p.sc[k].blocks;
  }
  OSVOS_CHECK_CUDA(ensure_dynamic_smem<side_folded_wgrad_kernel>(kSwSmemBytes));
  OSVOS_CHECK_CUDA(launch_pdl(side_folded_wgrad_kernel, dim3(begin), dim3(kSwKernelThreads), kSwSmemBytes,
                              static_cast<cudaStream_t>(stream_), maps, p));
  return OSVOS_OK;
}

extern "C" int osvos_side_folded_wgrad(const void* x_hi, const void* x_lo, const float* dpq, float* g, int n, int h,
                                       int w, int c, osvos_stream_t stream_) {
  osvos_side_wgrad_item it;
  it.x_hi = x_hi;
  it.x_lo = x_lo;
  it.dpq = dpq;
  it.g = g;
  it.n = n;
  it.h = h;
  it.w = w;
  it.c = c;
  return osvos_side_folded_wgrad_multi(&it, 1, stream_);
}

extern "C" int osvos_side_grads_finish(const osvos_side_grads_item* items, int count, osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(items != nullptr && count > 0 && count <= 4);
  SideGradTable t;
  t.count = count;
  for (int i = 0; i < count; ++i) {
    const osvos_side_grads_item& it = items[i];
    OSVOS_CHECK_ARG(it.g != nullptr && it.side_w != nullptr && it.proj_w != nullptr && it.d_side_w != nullptr &&
                    it.d_side_b != nullptr && it.c > 0);
    SideGradScale& L = t.s[i];
    L.g = it.g;
    L.side_w = it.side_w;
    L.side_b = it.side_b;
    L.proj = it.proj_w;
    L.d_side_w = it.d_side_w;
    L.d_side_b = it.d_side_b;
    L.d_score_w = it.d_score_w;
    L.d_score_b = it.d_score_b;
    L.d_fuse_w = it.d_fuse_w;
    L.c = it.c;
    L.accumulate = it.accumulate ? 1 : 0;
  }
  int cmax = 0;
  for (int i = 0; i < count; ++i) cmax = items[i].c > cmax ? items[i].c : cmax;
  OSVOS_CHECK_ARG(cmax <= 2048);
  const size_t smem = (static_cast<size_t>(18) * (cmax + 1) + 2) * sizeof(float);
  if (smem > 48 * 1024)
    OSVOS_CHECK_CUDA(ensure_dynamic_smem<side_grads_finish_kernel>((18 * 2049 + 2) * static_cast<int>(sizeof(float))));
  OSVOS_CHECK_CUDA(launch_pdl(side_grads_finish_kernel, dim3(16 * count), dim3(kFinThreads), smem, static_cast<cudaStream_t>(stream_), t));
  return OSVOS_OK;
}
