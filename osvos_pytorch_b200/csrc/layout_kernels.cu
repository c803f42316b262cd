// Bandwidth-bound helper kernels around the tensor-core convolutions:
// weight packing, NCHW<->act conversion, conv1_1 (Cin = 3), 2x2 ceil-mode max
// pooling, a CUDA-core reference conv (debug cross-check) and the standalone
// side-feature projection.
#include "common.cuh"

namespace osvos {

int conv_first_tc_launch(const float* x, const float* w_oihw, const float* bias, void* y_hi, void* y_lo, int n, int h,
                         int w, int flags, cudaStream_t stream);

// ------------------------------------------------------------ weight packing
// out[plane][tap][row][colp]; see include/osvos_b200.h.
__global__ void pack_weights_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int cout, int cin,
                                    int rows, int cols, int colp, int transpose_flip) {
  const size_t plane = static_cast<size_t>(9) * rows * colp;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < plane;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int col = static_cast<int>(i % colp);
    const int row = static_cast<int>((i / colp) % rows);
    const int tap = static_cast<int>(i / (static_cast<size_t>(colp) * rows));
    float v = 0.f;
    if (col < cols) {
      const int co = transpose_flip ? col : row;
      const int ci = transpose_flip ? row : col;
      const int t = transpose_flip ? 8 - tap : tap;
      v = w[(static_cast<size_t>(co) * cin + ci) * 9 + t];
    }
    __nv_bfloat16 hi, lo;
    split_bf16(v, hi, lo);
    out[i] = hi;
    out[plane + i] = lo;
  }
}

// ------------------------------------------------------------ folded side branch
// side_prep (3x3, C -> 16, no ReLU) followed by the two 1x1 projections (score_dsn; this scale's slice of fuse) is one
// linear 3x3 convolution C -> 2 (networks/vgg_osvos.py:41,44,54 run at :67,69,72):
//   W'[o][ci][tap] = sum_co proj_w[16 o + co] * w_side[co][ci][tap],  b'[o] = (o == 0 ? proj_b : 0) + sum_co proj_w[16 o + co] * b_side[co]
// written straight in the packed split-bf16 operand layout [plane][tap][o][ci] the side kernel's weight box reads.
__global__ void fold_side_weights_kernel(const float* __restrict__ w_side, const float* __restrict__ b_side,
                                         const float* __restrict__ proj_w, const float* __restrict__ proj_b,
                                         __nv_bfloat16* __restrict__ out, float* __restrict__ bias2, int cin) {
  const int plane = 9 * 2 * cin;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < plane; i += gridDim.x * blockDim.x) {
    const int ci = i % cin;
    const int o = (i / cin) & 1;
    const int tap = i / (2 * cin);
    float v = 0.f;
#pragma unroll
    for (int co = 0; co < 16; ++co) v = fmaf(__ldg(proj_w + 16 * o + co), __ldg(w_side + (static_cast<size_t>(co) * cin + ci) * 9 + tap), v);
    __nv_bfloat16 hi, lo;
    split_bf16(v, hi, lo);
    out[i] = hi;
    out[plane + i] = lo;
  }
  if (blockIdx.x == 0 && threadIdx.x < 2) {
    const int o = threadIdx.x;
    float b = (o == 0 && proj_b) ? __ldg(proj_b) : 0.f;
    if (b_side) {
      for (int co = 0; co < 16; ++co) b = fmaf(__ldg(proj_w + 16 * o + co), __ldg(b_side + co), b);
    }
    bias2[o] = b;
  }
}

// All scales of the side branch in ONE launch (training re-folds after every optimizer step), optionally with an fp32
// copy of W' in the same [tap][o][ci] order for the folded backward (side_bwd_folded.cu, bwd_kernels.cu).
struct FoldScale {
  const float* side_w;
  const float* side_b;
  const float* proj_w;
  const float* proj_b;
  __nv_bfloat16* packed;
  float* bias2;
  float* folded_f32;
  int cin;
  int begin;      // first index of this scale in the concatenated [18 * cin] index space
};
struct FoldTable {
  FoldScale s[4];
  int count;
  int total;
};
__global__ void fold_side_weights_multi_kernel(const __grid_constant__ FoldTable t) {
  for (int gi = blockIdx.x * blockDim.x + threadIdx.x; gi < t.total; gi += gridDim.x * blockDim.x) {
    int k = 0;
    while (k + 1 < t.count && gi >= t.s[k + 1].begin) ++k;
    const FoldScale& L = t.s[k];
    const int i = gi - L.begin, cin = L.cin, plane = 18 * cin;
    const int ci = i % cin;
    const int o = (i / cin) & 1;
    const int tap = i / (2 * cin);
    float v = 0.f;
#pragma unroll
    for (int co = 0; co < 16; ++co)
      v = fmaf(__ldg(L.proj_w + 16 * o + co), __ldg(L.side_w + (static_cast<size_t>(co) * cin + ci) * 9 + tap), v);
    __nv_bfloat16 hi, lo;
    split_bf16(v, hi, lo);
    L.packed[i] = hi;
    L.packed[plane + i] = lo;
    if (L.folded_f32) L.folded_f32[i] = v;
    if (i < 2) {
      float b = (i == 0 && L.proj_b) ? __ldg(L.proj_b) : 0.f;
      if (L.side_b) {
        for (int co = 0; co < 16; ++co) b = fmaf(__ldg(L.proj_w + 16 * i + co), __ldg(L.side_b + co), b);
      }
      L.bias2[i] = b;
    }
  }
}

// ------------------------------------------------------------ NCHW <-> act
__global__ void nchw_to_act_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ hi,
                                   __nv_bfloat16* __restrict__ lo, int n, int c, int h, int w) {
  const size_t total = static_cast<size_t>(n) * c * h * w;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ch = static_cast<int>(i % c);
    size_t pix = i / c;
    const int xx = static_cast<int>(pix % w);
    pix /= w;
    const int yy = static_cast<int>(pix % h);
    const int nn = static_cast<int>(pix / h);
    const float v = x[((static_cast<size_t>(nn) * c + ch) * h + yy) * w + xx];
    __nv_bfloat16 a, b;
    split_bf16(v, a, b);
    hi[i] = a;
    if (lo) lo[i] = b;
  }
}

__global__ void act_to_nchw_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo,
                                   float* __restrict__ y, int n, int c, int h, int w) {
  const size_t total = static_cast<size_t>(n) * c * h * w;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int xx = static_cast<int>(i % w);
    size_t r = i / w;
    const int yy = static_cast<int>(r % h);
    r /= h;
    const int ch = static_cast<int>(r % c);
    const int nn = static_cast<int>(r / c);
    const size_t src = ((static_cast<size_t>(nn) * h + yy) * w + xx) * c + ch;
    y[i] = __bfloat162float(hi[src]) + (lo ? __bfloat162float(lo[src]) : 0.f);
  }
}

// ---------------------------------------------------- conv1_1 (3 -> 64) + ReLU
// One thread per output pixel, 64 fp32 accumulators, weights broadcast from
// shared memory as [k = ci*9 + tap][co].  Input read straight from the caller's
// NCHW fp32 frame (coalesced along x).
constexpr int kFirstThreads = 128;
__global__ void __launch_bounds__(kFirstThreads)
conv_first_kernel(const float* __restrict__ x, const float* __restrict__ wgt, const float* __restrict__ bias,
                  __nv_bfloat16* __restrict__ y_hi, __nv_bfloat16* __restrict__ y_lo, int n, int h, int w, int relu) {
  __shared__ __align__(16) float ws[27 * 64];
  __shared__ float bs[64];
  for (int i = threadIdx.x; i < 27 * 64; i += kFirstThreads) {
    const int co = i & 63, k = i >> 6;  // ws[k][co] = w[co][ci][r][s], k = ci*9 + 3r + s
    ws[i] = wgt[co * 27 + k];
  }
  if (threadIdx.x < 64) bs[threadIdx.x] = bias ? bias[threadIdx.x] : 0.f;
  __syncthreads();
  const int xx = blockIdx.x * kFirstThreads + threadIdx.x;
  const int yy = blockIdx.y;
  const int nn = blockIdx.z;
  if (xx >= w) return;
  float in[27];
#pragma unroll
  for (int ci = 0; ci < 3; ++ci) {
    const float* plane = x + (static_cast<size_t>(nn) * 3 + ci) * h * w;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int iy = yy + r - 1;
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int ix = xx + s - 1;
        in[ci * 9 + r * 3 + s] = (iy >= 0 && iy < h && ix >= 0 && ix < w) ? __ldg(plane + static_cast<size_t>(iy) * w + ix) : 0.f;
      }
    }
  }
  const size_t pix = (static_cast<size_t>(nn) * h + yy) * w + xx;
#pragma unroll 1
  for (int c0 = 0; c0 < 64; c0 += 16) {
    float acc[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) acc[j] = bs[c0 + j];
#pragma unroll
    for (int k = 0; k < 27; ++k) {
      const float4* wr = reinterpret_cast<const float4*>(ws + k * 64 + c0);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 wv = wr[j];
        acc[4 * j + 0] = fmaf(in[k], wv.x, acc[4 * j + 0]);
        acc[4 * j + 1] = fmaf(in[k], wv.y, acc[4 * j + 1]);
        acc[4 * j + 2] = fmaf(in[k], wv.z, acc[4 * j + 2]);
        acc[4 * j + 3] = fmaf(in[k], wv.w, acc[4 * j + 3]);
      }
    }
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float a = acc[2 * j], b = acc[2 * j + 1];
      if (relu) {
        a = fmaxf(a, 0.f);
        b = fmaxf(b, 0.f);
      }
      __nv_bfloat16 h0, l0, h1, l1;
      split_bf16(a, h0, l0);
      split_bf16(b, h1, l1);
      hi[j] = pack_bf16x2(h0, h1);
      lo[j] = pack_bf16x2(l0, l1);
    }
    uint4* dh = reinterpret_cast<uint4*>(y_hi + pix * 64 + c0);
    dh[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    dh[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
    if (y_lo) {
      uint4* dl = reinterpret_cast<uint4*>(y_lo + pix * 64 + c0);
      dl[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      dl[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
    }
  }
}

// --------------------------------------- MaxPool2d(2, 2, ceil_mode=True) on act
// One thread per (output pixel, group of 8 channels): 16-byte loads/stores.
// The window is clipped at the bottom/right edge (ceil mode); ties keep the
// first element in (dy, dx) scan order, like torch's kernel.
__global__ void maxpool_kernel(const __nv_bfloat16* __restrict__ x_hi, const __nv_bfloat16* __restrict__ x_lo,
                               __nv_bfloat16* __restrict__ y_hi, __nv_bfloat16* __restrict__ y_lo, int n, int h, int w,
                               int c, int oh, int ow) {
  const int groups = c / 8;
  const size_t total = static_cast<size_t>(n) * oh * ow * groups;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(i % groups);
    size_t r = i / groups;
    const int ox = static_cast<int>(r % ow);
    r /= ow;
    const int oy = static_cast<int>(r % oh);
    const int nn = static_cast<int>(r / oh);
    float best[8];
    uint32_t bh[4] = {0, 0, 0, 0}, bl[4] = {0, 0, 0, 0};
    bool first = true;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int iy = 2 * oy + dy, ix = 2 * ox + dx;
        if (iy >= h || ix >= w) continue;
        const size_t src = ((static_cast<size_t>(nn) * h + iy) * w + ix) * c + g * 8;
        const uint4 vh = __ldg(reinterpret_cast<const uint4*>(x_hi + src));
        uint4 vl = make_uint4(0, 0, 0, 0);
        if (x_lo) vl = __ldg(reinterpret_cast<const uint4*>(x_lo + src));
        const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w};
        const uint32_t lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float v0 = bf16_lo_to_float(hw[t]) + bf16_lo_to_float(lw[t]);
          const float v1 = bf16_hi_to_float(hw[t]) + bf16_hi_to_float(lw[t]);
          if (first || v0 > best[2 * t]) {
            best[2 * t] = v0;
            bh[t] = (bh[t] & 0xFFFF0000u) | (hw[t] & 0xFFFFu);
            bl[t] = (bl[t] & 0xFFFF0000u) | (lw[t] & 0xFFFFu);
          }
          if (first || v1 > best[2 * t + 1]) {
            best[2 * t + 1] = v1;
            bh[t] = (bh[t] & 0xFFFFu) | (hw[t] & 0xFFFF0000u);
            bl[t] = (bl[t] & 0xFFFFu) | (lw[t] & 0xFFFF0000u);
          }
        }
        first = false;
      }
    }
    const size_t dst = ((static_cast<size_t>(nn) * oh + oy) * ow + ox) * c + g * 8;
    *reinterpret_cast<uint4*>(y_hi + dst) = make_uint4(bh[0], bh[1], bh[2], bh[3]);
    if (y_lo) *reinterpret_cast<uint4*>(y_lo + dst) = make_uint4(bl[0], bl[1], bl[2], bl[3]);
  }
}

// ------------------------------------------------ CUDA-core conv (debug check)
__global__ void conv3x3_simt_kernel(const __nv_bfloat16* __restrict__ x_hi, const __nv_bfloat16* __restrict__ x_lo,
                                    const __nv_bfloat16* __restrict__ wp, const float* __restrict__ bias,
                                    __nv_bfloat16* __restrict__ y_hi, __nv_bfloat16* __restrict__ y_lo,
                                    float* __restrict__ y_f32, const __nv_bfloat16* __restrict__ mask_hi, int n, int h,
                                    int w, int cin, int cout, int flags) {
  const size_t plane = static_cast<size_t>(9) * cout * cin;
  const size_t total = static_cast<size_t>(n) * h * w * cout;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int co = static_cast<int>(i % cout);
    size_t pix = i / cout;
    const int xx = static_cast<int>(pix % w);
    const int yy = static_cast<int>((pix / w) % h);
    const int nn = static_cast<int>(pix / (static_cast<size_t>(w) * h));
    float acc = bias ? bias[co] : 0.f;
    for (int tap = 0; tap < 9; ++tap) {
      const int iy = yy + tap / 3 - 1, ix = xx + tap % 3 - 1;
      if (iy < 0 || iy >= h || ix < 0 || ix >= w) continue;
      const size_t xs = ((static_cast<size_t>(nn) * h + iy) * w + ix) * cin;
      const size_t wsb = (static_cast<size_t>(tap) * cout + co) * cin;
      for (int ci = 0; ci < cin; ++ci) {
        const float xh = __bfloat162float(x_hi[xs + ci]);
        const float wh = __bfloat162float(wp[wsb + ci]);
        if (flags & OSVOS_FLAG_FAST) {
          acc = fmaf(xh, wh, acc);
        } else {
          const float xl = __bfloat162float(x_lo[xs + ci]);
          const float wl = __bfloat162float(wp[plane + wsb + ci]);
          acc = fmaf(xl, wh, acc);
          acc = fmaf(xh, wl, acc);
          acc = fmaf(xh, wh, acc);
        }
      }
    }
    if (flags & OSVOS_FLAG_RELU) acc = fmaxf(acc, 0.f);
    if ((flags & OSVOS_FLAG_RELU_MASK) && !(__bfloat162float(mask_hi[i]) > 0.f)) acc = 0.f;
    if (y_f32) y_f32[i] = acc;
    if (y_hi) {
      __nv_bfloat16 a, b;
      split_bf16(acc, a, b);
      y_hi[i] = a;
      if (y_lo) y_lo[i] = b;
    }
  }
}

__global__ void side_project_kernel(const float* __restrict__ feat, const float* __restrict__ pw,
                                    const float* __restrict__ pb, float* __restrict__ pq, size_t npix) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < npix;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float4* f = reinterpret_cast<const float4*>(feat + i * 16);
    float sp = pb ? __ldg(pb) : 0.f, sq = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 v = __ldg(f + j);
      sp = fmaf(v.x, __ldg(pw + 4 * j + 0), sp);
      sp = fmaf(v.y, __ldg(pw + 4 * j + 1), sp);
      sp = fmaf(v.z, __ldg(pw + 4 * j + 2), sp);
      sp = fmaf(v.w, __ldg(pw + 4 * j + 3), sp);
      sq = fmaf(v.x, __ldg(pw + 16 + 4 * j + 0), sq);
      sq = fmaf(v.y, __ldg(pw + 16 + 4 * j + 1), sq);
      sq = fmaf(v.z, __ldg(pw + 16 + 4 * j + 2), sq);
      sq = fmaf(v.w, __ldg(pw + 16 + 4 * j + 3), sq);
    }
    *reinterpret_cast<float2*>(pq + i * 2) = make_float2(sp, sq);
  }
}

static inline int grid_for(size_t total, int threads) {
  size_t blocks = (total + threads - 1) / threads;
  const size_t cap = static_cast<size_t>(device_sm_count()) * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

}  // namespace osvos

using namespace osvos;

extern "C" size_t osvos_packed_weight_bytes(int rows, int cols_padded) {
  return static_cast<size_t>(2) * 9 * rows * cols_padded * sizeof(__nv_bfloat16);
}

extern "C" int osvos_pack_conv3x3_weights(const float* w, void* packed, int cout, int cin, int transpose_flip,
                                          int col_pad, osvos_stream_t stream) {
  OSVOS_CHECK_ARG(w != nullptr && packed != nullptr && cout > 0 && cin > 0 && col_pad > 0);
  const int rows = transpose_flip ? cin : cout;
  const int cols = transpose_flip ? cout : cin;
  const int colp = (cols + col_pad - 1) / col_pad * col_pad;
  const size_t plane = static_cast<size_t>(9) * rows * colp;
  pack_weights_kernel<<<grid_for(plane, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w, static_cast<__nv_bfloat16*>(packed), cout, cin, rows, cols, colp, transpose_flip);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" int osvos_fold_side_weights(const float* side_w, const float* side_b, const float* proj_w, const float* proj_b,
                                       void* packed, float* bias2, int cin, osvos_stream_t stream) {
  OSVOS_CHECK_ARG(side_w != nullptr && proj_w != nullptr && packed != nullptr && bias2 != nullptr);
  OSVOS_CHECK_ARG(cin >= 64 && cin % 64 == 0);
  fold_side_weights_kernel<<<grid_for(static_cast<size_t>(18) * cin, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      side_w, side_b, proj_w, proj_b, static_cast<__nv_bfloat16*>(packed), bias2, cin);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" int osvos_fold_side_weights_multi(const osvos_fold_item* items, int count, osvos_stream_t stream) {
  OSVOS_CHECK_ARG(items != nullptr && count > 0 && count <= 4);
  FoldTable t;
  t.count = count;
  int total = 0;
  for (int k = 0; k < count; ++k) {
    const osvos_fold_item& it = items[k];
    OSVOS_CHECK_ARG(it.side_w != nullptr && it.proj_w != nullptr && it.packed != nullptr && it.bias2 != nullptr);
    OSVOS_CHECK_ARG(it.cin >= 64 && it.cin % 64 == 0 && it.cin <= 4096);
    FoldScale& L = t.s[k];
    L.side_w = it.side_w;
    L.side_b = it.side_b;
    L.proj_w = it.proj_w;
    L.proj_b = it.proj_b;
    L.packed = static_cast<__nv_bfloat16*>(it.packed);
    L.bias2 = it.bias2;
    L.folded_f32 = it.folded_f32;
    L.cin = it.cin;
    L.begin = total;
    total += 18 * it.cin;
  }
  t.total = total;
  fold_side_weights_multi_kernel<<<grid_for(static_cast<size_t>(total), 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(t);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" int osvos_nchw_to_act(const float* x, void* hi, void* lo, int n, int c, int h, int w,
                                 osvos_stream_t stream) {
  OSVOS_CHECK_ARG(x != nullptr && hi != nullptr && n > 0 && c > 0 && h > 0 && w > 0);
  const size_t total = static_cast<size_t>(n) * c * h * w;
  nchw_to_act_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, static_cast<__nv_bfloat16*>(hi), static_cast<__nv_bfloat16*>(lo), n, c, h, w);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" int osvos_act_to_nchw(const void* hi, const void* lo, float* y, int n, int c, int h, int w,
                                 osvos_stream_t stream) {
  OSVOS_CHECK_ARG(y != nullptr && hi != nullptr && n > 0 && c > 0 && h > 0 && w > 0);
  const size_t total = static_cast<size_t>(n) * c * h * w;
  act_to_nchw_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(hi), static_cast<const __nv_bfloat16*>(lo), y, n, c, h, w);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" int osvos_conv_first_fwd(const float* x, const float* w_oihw, const float* bias, void* y_hi, void* y_lo,
                                    int n, int h, int w, int flags, osvos_stream_t stream) {
  OSVOS_CHECK_ARG(x != nullptr && w_oihw != nullptr && y_hi != nullptr && n > 0 && h > 0 && w > 0);
  OSVOS_CHECK_ARG(h <= 65535 && n <= 65535);
  // the tensor-core kernel (conv_first_tc.cu), unless OSVOS_FIRST_IMPL=simt selects the CUDA-core one as a cross-check
  if (!env_is("OSVOS_FIRST_IMPL", "simt"))
    return conv_first_tc_launch(x, w_oihw, bias, y_hi, y_lo, n, h, w, flags, static_cast<cudaStream_t>(stream));
  dim3 grid((w + kFirstThreads - 1) / kFirstThreads, h, n);
  conv_first_kernel<<<grid, kFirstThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x, w_oihw, bias, static_cast<__nv_bfloat16*>(y_hi),
      (flags & OSVOS_FLAG_FAST) ? nullptr : static_cast<__nv_bfloat16*>(y_lo), n, h, w,
      (flags & OSVOS_FLAG_RELU) ? 1 : 0);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" int osvos_maxpool2x2_fwd(const void* x_hi, const void* x_lo, void* y_hi, void* y_lo, int n, int h, int w,
                                    int c, osvos_stream_t stream) {
  OSVOS_CHECK_ARG(x_hi != nullptr && y_hi != nullptr && n > 0 && h > 0 && w > 0 && c > 0 && c % 8 == 0);
  OSVOS_CHECK_ARG((x_lo == nullptr) == (y_lo == nullptr));
  const int oh = (h + 1) / 2, ow = (w + 1) / 2;
  const size_t total = static_cast<size_t>(n) * oh * ow * (c / 8);
  maxpool_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x_hi), static_cast<const __nv_bfloat16*>(x_lo),
      static_cast<__nv_bfloat16*>(y_hi), static_cast<__nv_bfloat16*>(y_lo), n, h, w, c, oh, ow);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" int osvos_conv3x3_simt(const osvos_conv3x3_args* a, osvos_stream_t stream) {
  OSVOS_CHECK_ARG(a != nullptr && a->x_hi != nullptr && a->w_packed != nullptr);
  OSVOS_CHECK_ARG((a->flags & OSVOS_FLAG_FAST) || a->x_lo != nullptr);
  OSVOS_CHECK_ARG(a->pq == nullptr && a->pool_hi == nullptr && a->colsum == nullptr);
  const size_t total = static_cast<size_t>(a->n) * a->h * a->w * a->cout;
  conv3x3_simt_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(a->x_hi), static_cast<const __nv_bfloat16*>(a->x_lo),
      static_cast<const __nv_bfloat16*>(a->w_packed), a->bias, static_cast<__nv_bfloat16*>(a->y_hi),
      static_cast<__nv_bfloat16*>(a->y_lo), a->y_f32, static_cast<const __nv_bfloat16*>(a->mask_hi), a->n, a->h, a->w,
      a->cin, a->cout, a->flags);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}

extern "C" int osvos_side_project(const float* feat, const float* proj_w, const float* proj_b, float* pq, int n, int h,
                                  int w, osvos_stream_t stream) {
  OSVOS_CHECK_ARG(feat != nullptr && proj_w != nullptr && pq != nullptr && n > 0 && h > 0 && w > 0);
  const size_t npix = static_cast<size_t>(n) * h * w;
  side_project_kernel<<<grid_for(npix, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(feat, proj_w, proj_b, pq,
                                                                                          npix);
  OSVOS_CHECK_CUDA(cudaGetLastError());
  return OSVOS_OK;
}
