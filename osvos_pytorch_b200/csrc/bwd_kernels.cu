// Bandwidth-bound backward kernels around the tensor-core dgrad / wgrad GEMMs:
// max-unpool + ReLU mask (+ the side branch's folded gradient), per-channel
// bias-gradient sums and the conv1_1 (Cin = 3) backward.
// They replace the autograd graph PyTorch builds for reference
// networks/vgg_osvos.py:59-74 (triggered at train_online.py:141, train_parent.py:164).
#include "common.cuh"
#include "ptx.cuh"

namespace osvos {

// (the adjoint of the bilinear tail lives in tail.cu, next to its forward)

// ---------------------------------------------------------------- generic sum
__global__ void __launch_bounds__(256) sum_f32_kernel(const float* __restrict__ x, size_t n, double* __restrict__ out,
                                                      float* __restrict__ result) {
  float acc = 0.f;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    acc += __ldg(x + i);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  __shared__ float red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += static_cast<double>(red[i]);
    atomicAdd(out, t);
  }
  // the last block to finish converts the fp64 total (out[1] holds the arrival counter)
  if (last_block_arrives(reinterpret_cast<unsigned int*>(out + 1)) && threadIdx.x == 0)
    result[0] = static_cast<float>(__ldcg(out));
}
__device__ __forceinline__ void load_pair8(const __nv_bfloat16* hi, const __nv_bfloat16* lo, size_t off, float (&v)[8]) {
  const uint4 vh = __ldg(reinterpret_cast<const uint4*>(hi + off));
  uint4 vl = make_uint4(0, 0, 0, 0);
  if (lo) vl = __ldg(reinterpret_cast<const uint4*>(lo + off));
  const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w};
  const uint32_t lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    v[2 * t] = bf16_lo_to_float(hw[t]) + bf16_lo_to_float(lw[t]);
    v[2 * t + 1] = bf16_hi_to_float(hw[t]) + bf16_hi_to_float(lw[t]);
  }
}

// dz = ReLU'(x) * (unpool(dpool) + side-branch gradient), + fused bias gradient (column sums).
// The side-branch gradient comes in one of two forms:
//   SIDE = false: `dside`, an fp32 map [n,h,w,c] (or none: stage 1 has no side branch);
//   SIDE = true:  the FOLDED form (side_bwd_folded.cu, eq. 2): dX[px][c] = sum_{t,o} W'[t][o][c] * dpq[px - t][o], formed on
//   the fly from the two projection gradients and the fp32 folded weights [9][2][c] - no map of the stage's size is written
//   or read for the side branch.  A thread owns 8 channels of the (up to) four pixels of a pooling window: the 4 x 4
//   window of dpq around them is loaded once (16 float2), and for each of the nine taps the 2 x 8 weights are fetched
//   ONCE and applied to all four pixels (64 FMAs per 4 vector loads).  `wsrc` is the table in shared memory when a block
//   has enough tiles to amortise copying it (18 c floats), else the table in global memory through L1.
// POOL = false: the deepest stage, whose output has no pooling consumer (dz = ReLU' * side gradient only).
template <bool POOL, bool SIDE>
__global__ void __launch_bounds__(256, SIDE ? 2 : 4)
unpool_add_mask_kernel(const __nv_bfloat16* __restrict__ dp_hi, const __nv_bfloat16* __restrict__ dp_lo,
                       const __nv_bfloat16* __restrict__ x_hi, const __nv_bfloat16* __restrict__ x_lo,
                       const float* __restrict__ dside, const float* __restrict__ dpq, const float* __restrict__ wfold,
                       __nv_bfloat16* __restrict__ dz_hi, __nv_bfloat16* __restrict__ dz_lo, float* __restrict__ colsum,
                       int n, int h, int w, int c, int oh, int ow, int wf_in_smem) {
  extern __shared__ float cs[];  // [c] block-local channel sums (fused bias gradient), then [18][c] folded weights
  float* wf = cs + c;
  if (colsum) {
    for (int i = threadIdx.x; i < c; i += blockDim.x) cs[i] = 0.f;
  }
  if (SIDE && wf_in_smem) {        // parameters, not the predecessor's output: may be read before pdl_wait
    for (int i = threadIdx.x; i < 18 * c; i += blockDim.x) wf[i] = __ldg(wfold + i);
  }
  __syncthreads();
  pdl_wait();               // dpool / dside / dpq are the previous kernels' outputs (ptx.cuh)
  pdl_launch_dependents();
  const float* wsrc = (SIDE && wf_in_smem) ? wf : wfold;
  const int groups = c / 8;
  // blockDim (256) is a multiple of `groups`: a thread keeps the same channel group over the whole loop, and a block
  // iteration covers 256 / groups consecutive (pooled) pixels of one row (32-bit index math only)
  const int g = static_cast<int>(threadIdx.x % groups);
  const int pl = static_cast<int>(threadIdx.x / groups);
  const int ppb = 256 / groups;
  const int tiles_x = (ow + ppb - 1) / ppb;
  const int total_tiles = n * oh * tiles_x;
  constexpr int kPos = POOL ? 4 : 1;
  constexpr int kWin = POOL ? 4 : 3;
  float csum[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    const int tx = tile % tiles_x, row = tile / tiles_x;
    const int oy = row % oh, nn = row / oh;
    const int ox = tx * ppb + pl;
    if (ox >= ow) continue;
    const int by = POOL ? 2 * oy : oy, bx = POOL ? 2 * ox : ox;     // first pixel of the window
    float ds[kPos][8];
#pragma unroll
    for (int q = 0; q < kPos; ++q)
#pragma unroll
      for (int j = 0; j < 8; ++j) ds[q][j] = 0.f;
    if (SIDE) {
      // dwin[u][v] = dpq[(by - 1 + u, bx - 1 + v)]; pixel (a, b) of the window and tap (r, s) meet at u = a + 2 - r,
      // v = b + 2 - s  (dpq[px - t], t = (r - 1, s - 1))
      float2 dwin[kWin][kWin];
      const float2* dq = reinterpret_cast<const float2*>(dpq) + static_cast<size_t>(nn) * h * w;
#pragma unroll
      for (int u = 0; u < kWin; ++u)
#pragma unroll
        for (int v = 0; v < kWin; ++v) {
          const int yy = by - 1 + u, xx = bx - 1 + v;
          dwin[u][v] = make_float2(0.f, 0.f);
          if (yy >= 0 && yy < h && xx >= 0 && xx < w) dwin[u][v] = __ldg(dq + yy * w + xx);
        }
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int s3 = 0; s3 < 3; ++s3) {
          const float* w0 = wsrc + (2 * (3 * r + s3)) * c + g * 8;
          const float4 a0 = *reinterpret_cast<const float4*>(w0), a1 = *reinterpret_cast<const float4*>(w0 + 4);
          const float4 b0 = *reinterpret_cast<const float4*>(w0 + c), b1 = *reinterpret_cast<const float4*>(w0 + c + 4);
#pragma unroll
          for (int q = 0; q < kPos; ++q) {
            const float2 d = dwin[(q >> 1) + 2 - r][(q & 1) + 2 - s3];
            ds[q][0] = fmaf(a0.x, d.x, fmaf(b0.x, d.y, ds[q][0]));
            ds[q][1] = fmaf(a0.y, d.x, fmaf(b0.y, d.y, ds[q][1]));
            ds[q][2] = fmaf(a0.z, d.x, fmaf(b0.z, d.y, ds[q][2]));
            ds[q][3] = fmaf(a0.w, d.x, fmaf(b0.w, d.y, ds[q][3]));
            ds[q][4] = fmaf(a1.x, d.x, fmaf(b1.x, d.y, ds[q][4]));
            ds[q][5] = fmaf(a1.y, d.x, fmaf(b1.y, d.y, ds[q][5]));
            ds[q][6] = fmaf(a1.z, d.x, fmaf(b1.z, d.y, ds[q][6]));
            ds[q][7] = fmaf(a1.w, d.x, fmaf(b1.w, d.y, ds[q][7]));
          }
        }
    }
    // pass 1: argmax (first maximum in (dy, dx) scan order) and positivity of the window elements
    float best[8];
    uint32_t arg = 0, pos = 0;  // arg: 2 bits per channel; pos: bit (q * 8 + j) = x[q][j] > 0
#pragma unroll
    for (int q = 0; q < kPos; ++q) {
      const int iy = by + (q >> 1), ix = bx + (q & 1);
      if (iy >= h || ix >= w) continue;
      float v[8];
      load_pair8(x_hi, x_lo, ((static_cast<size_t>(nn) * h + iy) * w + ix) * c + g * 8, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (q == 0 || v[j] > best[j]) {
          best[j] = v[j];
          arg = (arg & ~(3u << (2 * j))) | (static_cast<uint32_t>(q) << (2 * j));
        }
        if (v[j] > 0.f) pos |= 1u << (q * 8 + j);
      }
    }
    float dpv[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (POOL) load_pair8(dp_hi, dp_lo, ((static_cast<size_t>(nn) * oh + oy) * ow + ox) * c + g * 8, dpv);
    // pass 2: gradients of the window positions
#pragma unroll
    for (int q = 0; q < kPos; ++q) {
      const int iy = by + (q >> 1), ix = bx + (q & 1);
      if (iy >= h || ix >= w) continue;
      const size_t dst = ((static_cast<size_t>(nn) * h + iy) * w + ix) * c + g * 8;
      if (!SIDE && dside) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(dside + dst));
        const float4 b = __ldg(reinterpret_cast<const float4*>(dside + dst) + 1);
        ds[q][0] = a.x, ds[q][1] = a.y, ds[q][2] = a.z, ds[q][3] = a.w;
        ds[q][4] = b.x, ds[q][5] = b.y, ds[q][6] = b.z, ds[q][7] = b.w;
      }
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float v0 = ds[q][2 * t] + (((arg >> (4 * t)) & 3u) == static_cast<uint32_t>(q) ? dpv[2 * t] : 0.f);
        float v1 = ds[q][2 * t + 1] + (((arg >> (4 * t + 2)) & 3u) == static_cast<uint32_t>(q) ? dpv[2 * t + 1] : 0.f);
        if (!((pos >> (q * 8 + 2 * t)) & 1u)) v0 = 0.f;
        if (!((pos >> (q * 8 + 2 * t + 1)) & 1u)) v1 = 0.f;
        csum[2 * t] += v0;
        csum[2 * t + 1] += v1;
        __nv_bfloat16 h0, l0, h1, l1;
        split_bf16(v0, h0, l0);
        split_bf16(v1, h1, l1);
        hi[t] = pack_bf16x2(h0, h1);
        lo[t] = pack_bf16x2(l0, l1);
      }
      *reinterpret_cast<uint4*>(dz_hi + dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      if (dz_lo) *reinterpret_cast<uint4*>(dz_lo + dst) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
  }
  if (colsum) {
#pragma unroll
    for (int j = 0; j < 8; ++j) atomicAdd(&cs[g * 8 + j], csum[j]);
    __syncthreads();
    for (int i = threadIdx.x; i < c; i += blockDim.x) atomicAdd(colsum + i, cs[i]);
  }
}

// ------------------------------------------------- per-channel sums of an act
// out[c] += sum_px (hi + lo)[px][c]   (bias gradient; out zeroed by the caller)
__global__ void __launch_bounds__(256)
channel_sum_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo, size_t npix, int c,
                   float* __restrict__ out) {
  const int groups = c / 8;               // threads across channels (8 channels each)
  const int rows = 256 / groups;          // pixel rows handled concurrently by the block
  const int g = threadIdx.x % groups, ry = threadIdx.x / groups;
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (ry < rows) {
    for (size_t px = blockIdx.x * static_cast<size_t>(rows) + ry; px < npix; px += static_cast<size_t>(gridDim.x) * rows) {
      const uint4 vh = __ldg(reinterpret_cast<const uint4*>(hi + px * c + g * 8));
      uint4 vl = make_uint4(0, 0, 0, 0);
      if (lo) vl = __ldg(reinterpret_cast<const uint4*>(lo + px * c + g * 8));
      const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w};
      const uint32_t lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        acc[2 * t] += bf16_lo_to_float(hw[t]) + bf16_lo_to_float(lw[t]);
        acc[2 * t + 1] += bf16_hi_to_float(hw[t]) + bf16_hi_to_float(lw[t]);
      }
    }
  }
  extern __shared__ float sm[];  // [256][8]
#pragma unroll
  for (int j = 0; j < 8; ++j) sm[threadIdx.x * 8 + j] = acc[j];
  __syncthreads();
  for (int ch = threadIdx.x; ch < c; ch += 256) {
    const int gg = ch / 8, j = ch % 8;
    float t = 0.f;
    for (int r = 0; r < rows; ++r) t += sm[(r * groups + gg) * 8 + j];
    atomicAdd(out + ch, t);
  }
}

// -------------------------------------------------------------- conv1_1 bwd
// dW[co][ci][r][s] = sum_px dz[px][co] * x[ci][px + (r-1, s-1)]: a [32 (27 used) x 64] output with the whole image
// as reduction axis - 1.4 GFLOP at 480x854 against 105 MB of dz, i.e. HBM-bound once the arithmetic is cheap.  The
// tile is too thin for tcgen05 (N = 27), so the products run on warp-level mma.sync.m16n8k16 (bf16 in, fp32 acc):
//   C[k][co] += A[k][px] * B[px][co],  A = im2col rows of x (split into bf16 hi/lo here), B = dz (already hi/lo),
// three passes hi*hi + hi*lo + lo*hi like every other product of the path.  A chunk is 64 consecutive pixels of one
// image row: dz is copied 16 B at a time into padded rows (ldmatrix.trans reads them conflict-free), the 27 shifted
// row segments of x are coalesced loads with no index division.  Each of the 8 warps owns 8 output channels.
// (History: flat-pixel chunks + fp32 register tiles 146 us -> row chunks 103 us -> this kernel, see profiles/.)
constexpr int kFwPix = 64;
constexpr int kFwDzStride = 72;   // bf16 elements per smem row of a dz plane (64 + 8 pad -> 144 B, odd multiple of 16 B)
constexpr int kFwXStride = 72;    // bf16 elements per smem row of an im2col plane
constexpr int kFwCopies = 16;     // replicas of the partial result (atomic contention)
constexpr int kFwRawStride = 68;  // fp32 elements per staged source row (66 used)
// offset of im2col row k = ci*9 + r*3 + s inside the staged source rows: (ci*3 + r) * kFwRawStride + s
__constant__ int c_fw_koff[27] = {
    0 * 68 + 0, 0 * 68 + 1, 0 * 68 + 2, 1 * 68 + 0, 1 * 68 + 1, 1 * 68 + 2, 2 * 68 + 0, 2 * 68 + 1, 2 * 68 + 2,
    3 * 68 + 0, 3 * 68 + 1, 3 * 68 + 2, 4 * 68 + 0, 4 * 68 + 1, 4 * 68 + 2, 5 * 68 + 0, 5 * 68 + 1, 5 * 68 + 2,
    6 * 68 + 0, 6 * 68 + 1, 6 * 68 + 2, 7 * 68 + 0, 7 * 68 + 1, 7 * 68 + 2, 8 * 68 + 0, 8 * 68 + 1, 8 * 68 + 2};

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(static_cast<uint32_t>(__cvta_generic_to_shared(p))));
}
__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t (&r)[2], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];\n"
               : "=r"(r[0]), "=r"(r[1])
               : "r"(static_cast<uint32_t>(__cvta_generic_to_shared(p))));
}
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__global__ void __launch_bounds__(256)
conv_first_wgrad_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ dz_hi,
                        const __nv_bfloat16* __restrict__ dz_lo, float* __restrict__ dw, float* __restrict__ partial,
                        int n, int h, int w) {
  __shared__ __align__(16) __nv_bfloat16 dzs[2][kFwPix][kFwDzStride];   // [plane][px][co]
  __shared__ __align__(16) __nv_bfloat16 xs[2][32][kFwXStride];          // [plane][k][px]
  __shared__ float raw[9 * kFwRawStride];                                // [ci*3 + r][x0 - 1 + cc]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float acc[2][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int i = threadIdx.x; i < 2 * 5 * kFwXStride; i += 256)             // k = 27..31 are padding rows
    xs[i / (5 * kFwXStride)][27 + (i / kFwXStride) % 5][i % kFwXStride] = __float2bfloat16_rn(0.f);
  const int chunks_x = (w + kFwPix - 1) / kFwPix;
  const int total = n * h * chunks_x;
  const int planes = dz_lo ? 2 : 1;
  // Register double buffering: the global loads of tile i+1 (4 x 16 B of dz and up to 3 source pixels per thread) are
  // issued before the shared-memory work of tile i, so their latency overlaps the im2col expansion and the MMAs
  // (a single-buffered version spent half of its stall samples on the smem stores waiting for these loads).
  uint4 rdz[4];
  float rx[3];
  int valid = 0;
  auto fetch = [&](int tile) {
    const int cx = tile % chunks_x;
    const int row = tile / chunks_x;           // nn * h + yy
    const int yy = row % h, nn = row / h;
    const int x0 = cx * kFwPix;
    const int vld = min(kFwPix, w - x0);
    const size_t pbase = static_cast<size_t>(row) * w + x0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {              // dz: 2 planes x 64 px x 8 groups of 16 B
      const int i = threadIdx.x + 256 * u;
      const int pl = i >> 9, pp = (i >> 3) & 63, g = i & 7;
      rdz[u] = make_uint4(0, 0, 0, 0);
      if (pp < vld && pl < planes)
        rdz[u] = __ldg(reinterpret_cast<const uint4*>((pl ? dz_lo : dz_hi) + (pbase + pp) * 64 + g * 8));
    }
#pragma unroll
    for (int u = 0; u < 3; ++u) {              // the 9 source rows (3 channels x 3 dy), 66 pixels each
      const int e = threadIdx.x + 256 * u;
      const int rr = e / kFwRawStride, cc = e - rr * kFwRawStride;      // rr = ci * 3 + r
      const int ci = rr / 3, r = rr - ci * 3;
      const int iy = yy + r - 1, ix = x0 + cc - 1;
      rx[u] = 0.f;
      if (rr < 9 && cc < kFwPix + 2 && cc <= vld + 1 && iy >= 0 && iy < h && ix >= 0 && ix < w)
        rx[u] = __ldg(x + ((static_cast<size_t>(nn) * 3 + ci) * h + iy) * w + ix);
    }
    return vld;
  };
  int next_valid = blockIdx.x < total ? fetch(blockIdx.x) : 0;
  for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
    valid = next_valid;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = threadIdx.x + 256 * u;
      *reinterpret_cast<uint4*>(&dzs[i >> 9][(i >> 3) & 63][(i & 7) * 8]) = rdz[u];
    }
#pragma unroll
    for (int u = 0; u < 3; ++u) {
      const int e = threadIdx.x + 256 * u;
      if (e < 9 * kFwRawStride) raw[e] = rx[u];
    }
    if (tile + static_cast<int>(gridDim.x) < total) next_valid = fetch(tile + gridDim.x);
    __syncthreads();
    // ... expanded into the 27 im2col rows, split into bf16 hi / lo (a warp works on one k: uniform table index)
    {
      const int pp = threadIdx.x & 63, q = threadIdx.x >> 6;
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        const int k = q * 7 + j;
        if (k < 27) {
          const float v = pp < valid ? raw[c_fw_koff[k] + pp] : 0.f;
          __nv_bfloat16 hi, lo;
          split_bf16(v, hi, lo);
          xs[0][k][pp] = hi;
          xs[1][k][pp] = lo;
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < kFwPix / 16; ++ks) {
      uint32_t bh[2], bl[2];
      ldmatrix_x2_trans(bh, &dzs[0][16 * ks + (lane & 15)][8 * warp]);
      ldmatrix_x2_trans(bl, &dzs[1][16 * ks + (lane & 15)][8 * warp]);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        uint32_t ah[4], al[4];
        const int ar = mt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, ac = 16 * ks + (lane >> 4) * 8;
        ldmatrix_x4(ah, &xs[0][ar][ac]);
        ldmatrix_x4(al, &xs[1][ar][ac]);
        mma_bf16_16816(acc[mt], ah, bh);
        if (planes == 2) {
          mma_bf16_16816(acc[mt], ah, bl);
          mma_bf16_16816(acc[mt], al, bh);
        } else {
          mma_bf16_16816(acc[mt], al, bh);       // x keeps both halves even when dz is single-plane (fast mode)
        }
      }
    }
    __syncthreads();
  }
  // C fragment: rows g / g+8 (k), columns 2t, 2t+1 (co within the warp's 8 channels)
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = mt * 16 + g + (j >> 1) * 8;
      const int co = 8 * warp + 2 * t + (j & 1);
      // kFwCopies replicas of the 64 x 27 result spread the same-address atomic traffic of the blocks
      if (k < 27) atomicAdd(partial + (blockIdx.x % kFwCopies) * (64 * 27) + co * 27 + k, acc[mt][j]);
    }
  if (last_block_arrives(reinterpret_cast<unsigned int*>(partial + kFwCopies * 64 * 27))) {
    for (int i = threadIdx.x; i < 64 * 27; i += 256) {
      float t = 0.f;
#pragma unroll
      for (int c = 0; c < kFwCopies; ++c) t += __ldcg(partial + c * (64 * 27) + i);
      dw[i] = t;
    }
  }
}

// dx[ci][y][x] = sum_{r,s,co} dz[y - (r-1)][x - (s-1)][co] * w[co][ci][r][s]
__global__ void __launch_bounds__(128)
conv_first_dgrad_kernel(const __nv_bfloat16* __restrict__ dz_hi, const __nv_bfloat16* __restrict__ dz_lo,
                        const float* __restrict__ wgt, float* __restrict__ dx, int n, int h, int w) {
  __shared__ float ws[27 * 64];  // [k = ci*9 + r*3 + s][co]
  for (int i = threadIdx.x; i < 27 * 64; i += 128) {
    const int co = i & 63, k = i >> 6;
    ws[i] = wgt[co * 27 + k];
  }
  __syncthreads();
  const int xx = blockIdx.x * 128 + threadIdx.x, yy = blockIdx.y, nn = blockIdx.z;
  if (xx >= w) return;
  float acc[3] = {0.f, 0.f, 0.f};
  for (int r = 0; r < 3; ++r) {
    const int iy = yy - (r - 1);
    if (iy < 0 || iy >= h) continue;
    for (int s = 0; s < 3; ++s) {
      const int ix = xx - (s - 1);
      if (ix < 0 || ix >= w) continue;
      const size_t src = ((static_cast<size_t>(nn) * h + iy) * w + ix) * 64;
      const uint4* ph = reinterpret_cast<const uint4*>(dz_hi + src);
      const uint4* pl = dz_lo ? reinterpret_cast<const uint4*>(dz_lo + src) : nullptr;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint4 vh = __ldg(ph + j);
        uint4 vl = make_uint4(0, 0, 0, 0);
        if (pl) vl = __ldg(pl + j);
        const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w};
        const uint32_t lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float d0 = bf16_lo_to_float(hw[t]) + bf16_lo_to_float(lw[t]);
          const float d1 = bf16_hi_to_float(hw[t]) + bf16_hi_to_float(lw[t]);
          const int co = 8 * j + 2 * t;
#pragma unroll
          for (int ci = 0; ci < 3; ++ci) {
            const int k = ci * 9 + r * 3 + s;
            acc[ci] = fmaf(d0, ws[k * 64 + co], acc[ci]);
            acc[ci] = fmaf(d1, ws[k * 64 + co + 1], acc[ci]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int ci = 0; ci < 3; ++ci) dx[((static_cast<size_t>(nn) * 3 + ci) * h + yy) * w + xx] = acc[ci];
}

static inline int grid_cap(size_t blocks, int per_sm) {
  const size_t cap = static_cast<size_t>(device_sm_count()) * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

}  // namespace osvos

using namespace osvos;

extern "C" int osvos_sum_f32(const float* x, size_t n, double* scratch, float* out, osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(x != nullptr && scratch != nullptr && out != nullptr && n > 0);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  OSVOS_CHECK_CUDA(cudaMemsetAsync(scratch, 0, 2 * sizeof(double), stream));
  sum_f32_kernel<<<grid_cap((n + 255) / 256, 4), 256, 0, stream>>>(x, n, scratch, out);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

template <bool POOL, bool SIDE>
static int launch_unpool(const void* dpool_hi, const void* dpool_lo, const void* x_hi, const void* x_lo, const float* dside,
                         const float* dpq, const float* wfold, void* dz_hi, void* dz_lo, float* colsum, int n, int h, int w,
                         int c, cudaStream_t stream) {
  const int oh = POOL ? (h + 1) / 2 : h, ow = POOL ? (w + 1) / 2 : w;
  const int ppb = 256 / (c / 8);
  const size_t tiles = static_cast<size_t>(n) * oh * ((ow + ppb - 1) / ppb);
  OSVOS_CHECK_ARG(tiles < (static_cast<size_t>(1) << 31));
  const int grid = grid_cap(tiles, SIDE ? 2 : 4);
  // the folded weights go to shared memory when every block has tiles enough to amortise the copy
  const int wf_in_smem = (SIDE && tiles >= static_cast<size_t>(grid) * 4) ? 1 : 0;
  const size_t smem = static_cast<size_t>(c) * sizeof(float) * (wf_in_smem ? 19 : 1);
  constexpr auto kern = unpool_add_mask_kernel<POOL, SIDE>;
  if (smem > 48 * 1024) OSVOS_CHECK_CUDA(ensure_dynamic_smem<kern>(19 * 2048 * sizeof(float)));
  OSVOS_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(256), smem, stream,
                              static_cast<const __nv_bfloat16*>(dpool_hi), static_cast<const __nv_bfloat16*>(dpool_lo),
                              static_cast<const __nv_bfloat16*>(x_hi), static_cast<const __nv_bfloat16*>(x_lo), dside, dpq,
                              wfold, static_cast<__nv_bfloat16*>(dz_hi), static_cast<__nv_bfloat16*>(dz_lo), colsum, n, h, w,
                              c, oh, ow, wf_in_smem));
  return OSVOS_OK;
}

extern "C" int osvos_unpool_add_mask(const void* dpool_hi, const void* dpool_lo, const void* x_hi, const void* x_lo,
                                     const float* dside, void* dz_hi, void* dz_lo, float* colsum, int n, int h, int w,
                                     int c, osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(dpool_hi != nullptr && x_hi != nullptr && dz_hi != nullptr && n > 0 && h > 0 && w > 0 && c % 8 == 0);
  OSVOS_CHECK_ARG(c <= 2048 && 256 % (c / 8) == 0);
  return launch_unpool<true, false>(dpool_hi, dpool_lo, x_hi, x_lo, dside, nullptr, nullptr, dz_hi, dz_lo, colsum, n, h, w, c,
                             static_cast<cudaStream_t>(stream_));
}

extern "C" int osvos_unpool_side_mask(const void* dpool_hi, const void* dpool_lo, const void* x_hi, const void* x_lo,
                                      const float* dpq, const float* wfold, void* dz_hi, void* dz_lo, float* colsum, int n,
                                      int h, int w, int c, osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(x_hi != nullptr && dz_hi != nullptr && dpq != nullptr && wfold != nullptr && n > 0 && h > 0 && w > 0 &&
                  c % 8 == 0);
  OSVOS_CHECK_ARG(c <= 2048 && 256 % (c / 8) == 0);
  OSVOS_CHECK_ARG(static_cast<long>(h) * w < (1l << 30));
  OSVOS_CHECK_ARG((reinterpret_cast<uintptr_t>(wfold) & 15) == 0);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (dpool_hi != nullptr)
    return launch_unpool<true, true>(dpool_hi, dpool_lo, x_hi, x_lo, nullptr, dpq, wfold, dz_hi, dz_lo, colsum, n, h, w, c, stream);
  return launch_unpool<false, true>(nullptr, nullptr, x_hi, x_lo, nullptr, dpq, wfold, dz_hi, dz_lo, colsum, n, h, w, c, stream);
}

extern "C" int osvos_channel_sum(const void* act_hi, const void* act_lo, float* out, size_t npix, int c,
                                 osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(act_hi != nullptr && out != nullptr && npix > 0 && c % 8 == 0 && c >= 8 && c <= 2048 &&
                  256 % (c / 8) == 0);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  OSVOS_CHECK_CUDA(cudaMemsetAsync(out, 0, c * sizeof(float), stream));
  const int rows = 256 / (c / 8);
  const size_t blocks = (npix + rows - 1) / rows;
  channel_sum_kernel<<<grid_cap(blocks, 4), 256, 256 * 8 * sizeof(float), stream>>>(
      static_cast<const __nv_bfloat16*>(act_hi), static_cast<const __nv_bfloat16*>(act_lo), npix, c, out);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" size_t osvos_conv_first_bwd_workspace_bytes(void) { return (kFwCopies * 64 * 27 + 4) * sizeof(float); }

extern "C" int osvos_conv_first_bwd(const float* x_nchw, const void* dz_hi, const void* dz_lo, const float* w_oihw,
                                    float* dw, float* dx_nchw, void* workspace, int n, int h, int w,
                                    osvos_stream_t stream_) {
  OSVOS_CHECK_ARG(x_nchw != nullptr && dz_hi != nullptr && dw != nullptr && workspace != nullptr && n > 0 && h > 0 &&
                  w > 0);
  OSVOS_CHECK_ARG(dx_nchw == nullptr || w_oihw != nullptr);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  OSVOS_CHECK_CUDA(cudaMemsetAsync(workspace, 0, osvos_conv_first_bwd_workspace_bytes(), stream));
  const size_t tiles = static_cast<size_t>(n) * h * ((w + kFwPix - 1) / kFwPix);
  conv_first_wgrad_kernel<<<grid_cap(tiles, 4), 256, 0, stream>>>(
      x_nchw, static_cast<const __nv_bfloat16*>(dz_hi), static_cast<const __nv_bfloat16*>(dz_lo), dw,
      static_cast<float*>(workspace), n, h, w);
  if (dx_nchw) {
    dim3 grid((w + 127) / 128, h, n);
    conv_first_dgrad_kernel<<<grid, 128, 0, stream>>>(static_cast<const __nv_bfloat16*>(dz_hi),
                                                       static_cast<const __nv_bfloat16*>(dz_lo), w_oihw, dx_nchw, n, h,
                                                       w);
  }
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}
