// Conv trunk of the DQN (reference rainbowiqn/model.py:65-67,115-118) as im2col + GEMM.
//
//   conv1 8x8 s4 p1 (4->32)   conv2 4x4 s2 (32->64)   conv3 3x3 s1 (64->64), ReLU after each,
//   activations NCHW so that conv3's output flattens C-major into the 3136 features the
//   quantile embedding and the NoisyLinear head expect (model.py:118).
//
// The uint8 frame stack (B,4,84,84) is read directly: x = float(u8) / 255.0f reproduces the
// reference's `.to(float32).div_(255)` (redis_memory.py:527-536) bit for bit, without ever
// materialising the fp32 frames in HBM.
#include "common.cuh"
#include "gemm.h"
#include "../../include/riqn_b200.h"

namespace riqn {

template <typename T>
__device__ __forceinline__ float load_px(const T* p);
template <>
__device__ __forceinline__ float load_px<uint8_t>(const uint8_t* p) { return (float)(*p) / 255.0f; }
template <>
__device__ __forceinline__ float load_px<float>(const float* p) { return *p; }

// col[m, k] , m = (b, oh, ow), k = (cin, kh, kw)  -- k order == the (Cout, Cin*KH*KW) weight layout
template <typename T>
__global__ void im2col_kernel(riqn_conv_geom g, const T* __restrict__ in, float* __restrict__ col) {
  const int K = g.Cin * g.KH * g.KW;
  const long total = (long)g.B * g.OH * g.OW * K;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int k = (int)(idx % K);
    const long m = idx / K;
    const int kw = k % g.KW, kh = (k / g.KW) % g.KH, c = k / (g.KW * g.KH);
    const int ow = (int)(m % g.OW), oh = (int)((m / g.OW) % g.OH), b = (int)(m / ((long)g.OW * g.OH));
    const int ih = oh * g.stride + kh - g.pad, iw = ow * g.stride + kw - g.pad;
    float v = 0.f;
    if (ih >= 0 && ih < g.H && iw >= 0 && iw < g.W) v = load_px<T>(&in[(long)b * g.in_bstride + ((long)c * g.H + ih) * g.W + iw]);
    col[idx] = v;
  }
}

// dY[m, c] = dout[b, c, p] * (out[b, c, p] > 0)      (ReLU backward + NCHW -> (M, Cout))
__global__ void conv_dy_kernel(int B, int Cout, int ohw, const float* __restrict__ dout,
                               const float* __restrict__ out, float* __restrict__ dY) {
  const long total = (long)B * Cout * ohw;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int p = (int)(idx % ohw);
    const int c = (int)((idx / ohw) % Cout);
    const long b = idx / ((long)ohw * Cout);
    const float v = out[idx] > 0.f ? dout[idx] : 0.f;
    dY[(b * ohw + p) * Cout + c] = v;
  }
}

// din[b, c, ih, iw] = sum_{kh,kw} dcol[(b,oh,ow), (c,kh,kw)]
__global__ void col2im_kernel(riqn_conv_geom g, const float* __restrict__ dcol, float* __restrict__ din) {
  const int K = g.Cin * g.KH * g.KW;
  const long total = (long)g.B * g.Cin * g.H * g.W;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int iw = (int)(idx % g.W), ih = (int)((idx / g.W) % g.H);
    const int c = (int)((idx / ((long)g.W * g.H)) % g.Cin);
    const long b = idx / ((long)g.W * g.H * g.Cin);
    float acc = 0.f;
    for (int kh = 0; kh < g.KH; ++kh) {
      const int t = ih + g.pad - kh;
      if (t < 0 || t % g.stride) continue;
      const int oh = t / g.stride;
      if (oh >= g.OH) continue;
      for (int kw = 0; kw < g.KW; ++kw) {
        const int u = iw + g.pad - kw;
        if (u < 0 || u % g.stride) continue;
        const int ow = u / g.stride;
        if (ow >= g.OW) continue;
        acc += dcol[((b * g.OH + oh) * g.OW + ow) * K + (c * g.KH + kh) * g.KW + kw];
      }
    }
    din[idx] = acc;
  }
}

// Same scatter with coalesced reads: one block per (sample, chunk of CC input channels) streams that sample's dcol rows
// (the CC*KH*KW gradients of a row are contiguous) and accumulates into a shared-memory image tile, written out once.
__global__ void col2im_tile_kernel(riqn_conv_geom g, int CC, const float* __restrict__ dcol, float* __restrict__ din) {
  extern __shared__ float acc[];     // CC * H * W
  const int K = g.Cin * g.KH * g.KW, khw = g.KH * g.KW, ohw = g.OH * g.OW, hw = g.H * g.W;
  const int chunks = g.Cin / CC;
  const long b = blockIdx.x / chunks;
  const int c0 = (blockIdx.x % chunks) * CC;
  for (int i = threadIdx.x; i < CC * hw; i += blockDim.x) acc[i] = 0.f;
  __syncthreads();
  const int per_row = CC * khw;
  const float* base = dcol + b * ohw * (long)K + (long)c0 * khw;
  for (int e = threadIdx.x; e < ohw * per_row; e += blockDim.x) {
    const int m = e / per_row, j = e - m * per_row;
    const int c = j / khw, r = j - c * khw;
    const int kh = r / g.KW, kw = r - kh * g.KW;
    const int oh = m / g.OW, ow = m - oh * g.OW;
    const int ih = oh * g.stride + kh - g.pad, iw = ow * g.stride + kw - g.pad;
    if (ih >= 0 && ih < g.H && iw >= 0 && iw < g.W) atomicAdd(&acc[c * hw + ih * g.W + iw], base[(long)m * K + j]);
  }
  __syncthreads();
  float* out = din + (b * g.Cin + c0) * hw;
  for (int i = threadIdx.x; i < CC * hw; i += blockDim.x) out[i] = acc[i];
}

static int col2im(const riqn_conv_geom* g, const float* dcol, float* din, cudaStream_t s) {
  const int hw = g->H * g->W;
  int CC = g->Cin;
  while (CC > 1 && ((long)CC * hw * 4 > 16 * 1024 || g->Cin % CC)) --CC;
  if ((long)CC * hw * 4 <= 48 * 1024) {
    col2im_tile_kernel<<<g->B * (g->Cin / CC), 256, (size_t)CC * hw * 4, s>>>(*g, CC, dcol, din);
  } else {
    long total = (long)g->B * g->Cin * hw;
    long blocks = (total + 255) / 256;
    col2im_kernel<<<(int)(blocks > 148L * 32 ? 148L * 32 : blocks), 256, 0, s>>>(*g, dcol, din);
  }
  return (int)cudaGetLastError();
}

// out[n] += sum_m X[m, n]
__global__ void colsum_atomic_kernel(long M, int N, const float* __restrict__ X, float* __restrict__ out, int rows_per_block) {
  const int n = blockIdx.x * 128 + (threadIdx.x & 127);
  const int half = threadIdx.x >> 7;
  if (n >= N) return;
  const long r0 = (long)blockIdx.y * rows_per_block;
  const long r1 = min(M, r0 + rows_per_block);
  float acc = 0.f;
  for (long r = r0 + half; r < r1; r += 2) acc += X[r * N + n];
  atomicAdd(&out[n], acc);
}

int colsum_atomic(long M, int N, const float* X, float* out, cudaStream_t s) {
  int rows_per_block = 256;
  dim3 grid((N + 127) / 128, (unsigned)((M + rows_per_block - 1) / rows_per_block));
  colsum_atomic_kernel<<<grid, 256, 0, s>>>(M, N, X, out, rows_per_block);
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// Tensor-core path: im2col straight into bf16 (hi, lo) operands for gemm_tc.cu
// ---------------------------------------------------------------------------------------------------------------
using bf16 = __nv_bfloat16;

template <typename T>
__device__ __forceinline__ float im2col_at(const riqn_conv_geom& g, const T* __restrict__ in, long m, int k) {
  const int kw = k % g.KW, kh = (k / g.KW) % g.KH, c = k / (g.KW * g.KH);
  const int ow = (int)(m % g.OW), oh = (int)((m / g.OW) % g.OH);
  const long b = m / ((long)g.OW * g.OH);
  const int ih = oh * g.stride + kh - g.pad, iw = ow * g.stride + kw - g.pad;
  if (ih < 0 || ih >= g.H || iw < 0 || iw >= g.W) return 0.f;
  return load_px<T>(&in[b * g.in_bstride + ((long)c * g.H + ih) * g.W + iw]);
}

__device__ __forceinline__ void pack8(const float (&x)[8], uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int t = 0; t < 8; t += 2) {
    const bf16 h0 = __float2bfloat16_rn(x[t]), h1 = __float2bfloat16_rn(x[t + 1]);
    const bf16 l0 = __float2bfloat16_rn(x[t] - __bfloat162float(h0)), l1 = __float2bfloat16_rn(x[t + 1] - __bfloat162float(h1));
    h[t / 2] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
    l[t / 2] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// col (M, K): one thread = 8 consecutive k of one row m -> one 16-byte store per image.  (c, kh, kw) of the first
// k is decoded once and then stepped without divisions.
template <typename T>
__global__ void im2col_bf16_kernel(riqn_conv_geom g, const T* __restrict__ in, bf16* __restrict__ hi, bf16* __restrict__ lo) {
  const int K = g.Cin * g.KH * g.KW, K8 = K / 8;
  const long total = (long)g.B * g.OH * g.OW * K8;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int k0 = (int)(idx % K8) * 8;
    const long m = idx / K8;
    const int ow = (int)(m % g.OW), oh = (int)((m / g.OW) % g.OH);
    const long b = m / ((long)g.OW * g.OH);
    int kw = k0 % g.KW, kh = (k0 / g.KW) % g.KH, c = k0 / (g.KW * g.KH);
    const T* base = in + b * g.in_bstride;
    const int ih0 = oh * g.stride - g.pad, iw0 = ow * g.stride - g.pad;
    float x[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int ih = ih0 + kh, iw = iw0 + kw;
      x[t] = (ih >= 0 && ih < g.H && iw >= 0 && iw < g.W) ? load_px<T>(&base[((long)c * g.H + ih) * g.W + iw]) : 0.f;
      if (++kw == g.KW) { kw = 0; if (++kh == g.KH) { kh = 0; ++c; } }
    }
    uint4 h, l;
    pack8(x, h, l);
    *reinterpret_cast<uint4*>(hi + m * K + k0) = h;
    if (lo) *reinterpret_cast<uint4*>(lo + m * K + k0) = l;
  }
}

// uint8 specialisation: the 256 possible pixels are converted once per block into a packed (hi | lo << 16) table, so
// the per-element work is one byte load + one shared-memory lookup (bit-identical to x / 255.0f then hi/lo split).
__global__ void im2col_bf16_u8_kernel(riqn_conv_geom g, const uint8_t* __restrict__ in, bf16* __restrict__ hi, bf16* __restrict__ lo) {
  __shared__ uint32_t lut[256];
  {
    const float x = (float)threadIdx.x / 255.0f;
    const bf16 h = __float2bfloat16_rn(x);
    const bf16 l = __float2bfloat16_rn(x - __bfloat162float(h));
    if (threadIdx.x < 256) lut[threadIdx.x] = (uint32_t)__bfloat16_as_ushort(h) | ((uint32_t)__bfloat16_as_ushort(l) << 16);
  }
  __syncthreads();
  const int K = g.Cin * g.KH * g.KW, K8 = K / 8;
  const long total = (long)g.B * g.OH * g.OW * K8;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int k0 = (int)(idx % K8) * 8;
    const long m = idx / K8;
    const int ow = (int)(m % g.OW), oh = (int)((m / g.OW) % g.OH);
    const long b = m / ((long)g.OW * g.OH);
    int kw = k0 % g.KW, kh = (k0 / g.KW) % g.KH, c = k0 / (g.KW * g.KH);
    const uint8_t* base = in + b * g.in_bstride;
    const int ih0 = oh * g.stride - g.pad, iw0 = ow * g.stride - g.pad;
    uint32_t e[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int ih = ih0 + kh, iw = iw0 + kw;
      e[t] = (ih >= 0 && ih < g.H && iw >= 0 && iw < g.W) ? lut[base[((long)c * g.H + ih) * g.W + iw]] : 0u;
      if (++kw == g.KW) { kw = 0; if (++kh == g.KH) { kh = 0; ++c; } }
    }
    uint4 h, l;
    h.x = (e[0] & 0xffffu) | (e[1] << 16); h.y = (e[2] & 0xffffu) | (e[3] << 16);
    h.z = (e[4] & 0xffffu) | (e[5] << 16); h.w = (e[6] & 0xffffu) | (e[7] << 16);
    l.x = (e[0] >> 16) | (e[1] & 0xffff0000u); l.y = (e[2] >> 16) | (e[3] & 0xffff0000u);
    l.z = (e[4] >> 16) | (e[5] & 0xffff0000u); l.w = (e[6] >> 16) | (e[7] & 0xffff0000u);
    *reinterpret_cast<uint4*>(hi + m * K + k0) = h;
    if (lo) *reinterpret_cast<uint4*>(lo + m * K + k0) = l;
  }
}

// Raw-pixel im2col for the first layer: one block per sample stages the uint8 frame stack in shared memory (coalesced
// 16-byte loads), then writes col (M, K) -- and colT (K, M) for the backward -- with the pixel VALUES 0..255 as bf16
// (exact); the 1/255 of the reference (redis_memory.py:527-536) is folded into the weights / the gradient scale.
__global__ void im2col_u8_staged_kernel(riqn_conv_geom g, const uint8_t* __restrict__ in, bf16* __restrict__ col,
                                        bf16* __restrict__ colT) {
  extern __shared__ __align__(16) uint8_t img[];
  const int chw = g.Cin * g.H * g.W, K = g.Cin * g.KH * g.KW, K8 = K / 8, ohw = g.OH * g.OW;
  const long b = blockIdx.x;
  const int part = blockIdx.y, parts = gridDim.y;            // several blocks share a sample: more CTAs than SMs
  const uint4* src = reinterpret_cast<const uint4*>(in + b * g.in_bstride);
  for (int i = threadIdx.x; i < chw / 16; i += blockDim.x) reinterpret_cast<uint4*>(img)[i] = src[i];
  __syncthreads();
  auto px = [&](int c, int ih, int iw) -> uint32_t {
    if (ih < 0 || ih >= g.H || iw < 0 || iw >= g.W) return 0u;
    return __float_as_uint((float)img[(c * g.H + ih) * g.W + iw]) >> 16;     // exact bf16 bits of 0..255
  };
  // Fast path (the Atari first layer: 8-wide rows, stride 4, pad 1, nothing hangs over the right / bottom edge): a
  // kernel row is bytes 4*ow-1 .. 4*ow+6 of an image row = byte 3 of word ow-1, word ow, bytes 0..2 of word ow+1.
  const bool fast = g.KW == 8 && g.stride == 4 && g.pad == 1 && (g.W & 3) == 0 && (g.OW - 1) * 4 + 6 < g.W &&
                    (g.OH - 1) * 4 - 1 + g.KH - 1 < g.H;
  auto cvt2 = [](uint32_t w, uint32_t sa, uint32_t sb) -> uint32_t {      // two bytes of w -> two bf16 (exact)
    const float fa = __uint_as_float(__byte_perm(w, 0x4B000000u, sa)) - 8388608.0f;
    const float fb = __uint_as_float(__byte_perm(w, 0x4B000000u, sb)) - 8388608.0f;
    return __byte_perm(__float_as_uint(fa), __float_as_uint(fb), 0x7632);
  };
  if (col && fast) {
    const uint32_t* img32 = reinterpret_cast<const uint32_t*>(img);
    const int wpr = g.W >> 2;                                   // words per image row
    for (int item = part * blockDim.x + threadIdx.x; item < ohw * K8; item += parts * blockDim.x) {
      const int m = item / K8, kr = item - m * K8;              // kr = c * KH + kh
      const int oh = m / g.OW, ow = m - oh * g.OW;
      const int c = kr / g.KH, kh = kr - c * g.KH;
      const int ih = oh * 4 - 1 + kh;
      uint4 o = make_uint4(0u, 0u, 0u, 0u);
      if (ih >= 0) {
        const uint32_t* rowp = img32 + (c * g.H + ih) * wpr + ow;
        const uint32_t w0 = ow > 0 ? rowp[-1] : 0u, w1 = rowp[0], w2 = rowp[1];
        const uint32_t a = __byte_perm(w0, w1, 0x0043);          // bytes: w0.3, w1.0   (upper two unused)
        o.x = cvt2(a, 0x7650, 0x7651);
        o.y = cvt2(w1, 0x7651, 0x7652);
        o.z = cvt2(__byte_perm(w1, w2, 0x0043), 0x7650, 0x7651);
        o.w = cvt2(w2, 0x7651, 0x7652);
      }
      *reinterpret_cast<uint4*>(col + (b * ohw + m) * K + kr * 8) = o;
    }
  } else if (col) {
    for (int item = part * blockDim.x + threadIdx.x; item < ohw * K8; item += parts * blockDim.x) {
      const int m = item / K8, k0 = (item - m * K8) * 8;
      const int oh = m / g.OW, ow = m - oh * g.OW;
      int kw = k0 % g.KW, kh = (k0 / g.KW) % g.KH, c = k0 / (g.KW * g.KH);
      const int ih0 = oh * g.stride - g.pad, iw0 = ow * g.stride - g.pad;
      uint32_t e[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        e[t] = px(c, ih0 + kh, iw0 + kw);
        if (++kw == g.KW) { kw = 0; if (++kh == g.KH) { kh = 0; ++c; } }
      }
      *reinterpret_cast<uint4*>(col + (b * ohw + m) * K + k0) =
          make_uint4(e[0] | (e[1] << 16), e[2] | (e[3] << 16), e[4] | (e[5] << 16), e[6] | (e[7] << 16));
    }
  }
  if (colT) {
    const long M = (long)g.B * ohw;
    const int M8 = ohw / 8;
    for (int item = part * blockDim.x + threadIdx.x; item < K * M8; item += parts * blockDim.x) {
      const int k = item / M8, m0 = (item - k * M8) * 8;
      const int kw = k % g.KW, kh = (k / g.KW) % g.KH, c = k / (g.KW * g.KH);
      int oh = m0 / g.OW, ow = m0 - oh * g.OW;
      uint32_t e[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        e[t] = px(c, oh * g.stride + kh - g.pad, ow * g.stride + kw - g.pad);
        if (++ow == g.OW) { ow = 0; ++oh; }
      }
      *reinterpret_cast<uint4*>(colT + (long)k * M + b * ohw + m0) =
          make_uint4(e[0] | (e[1] << 16), e[2] | (e[3] << 16), e[4] | (e[5] << 16), e[6] | (e[7] << 16));
    }
  }
}

// fp32 NCHW input, staged: one block per sample converts its input ONCE into packed (hi | lo << 16) words in shared
// memory (coalesced 16-byte loads; the plain kernel converts every pixel KH*KW/stride^2 times), then assembles the
// (M, K) hi / lo rows from shared memory with 32-bit index arithmetic.  Bit-identical to im2col_bf16_kernel.
__global__ void __launch_bounds__(256) im2col_f32_staged_kernel(riqn_conv_geom g, const float* __restrict__ in,
                                                                bf16* __restrict__ hi, bf16* __restrict__ lo) {
  extern __shared__ __align__(16) uint32_t simg[];
  const int chw = g.Cin * g.H * g.W, K = g.Cin * g.KH * g.KW, K8 = K / 8, ohw = g.OH * g.OW;
  const long b = blockIdx.x;
  const float4* src = reinterpret_cast<const float4*>(in + b * g.in_bstride);
  for (int i = threadIdx.x; i < chw / 4; i += blockDim.x) {
    const float4 v = __ldg(src + i);
    const float x[4] = {v.x, v.y, v.z, v.w};
    uint32_t w[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const bf16 h = __float2bfloat16_rn(x[t]);
      const bf16 l = __float2bfloat16_rn(x[t] - __bfloat162float(h));
      w[t] = (uint32_t)__bfloat16_as_ushort(h) | ((uint32_t)__bfloat16_as_ushort(l) << 16);
    }
    reinterpret_cast<uint4*>(simg)[i] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  __syncthreads();
  const int hw = g.H * g.W;
  for (int item = threadIdx.x; item < ohw * K8; item += blockDim.x) {
    const int m = item / K8, k0 = (item - m * K8) * 8;
    const int oh = m / g.OW, ow = m - oh * g.OW;
    int kw = k0 % g.KW, kh = (k0 / g.KW) % g.KH, c = k0 / (g.KW * g.KH);
    const int ih0 = oh * g.stride - g.pad, iw0 = ow * g.stride - g.pad;
    uint32_t e[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int ih = ih0 + kh, iw = iw0 + kw;
      e[t] = ((unsigned)ih < (unsigned)g.H && (unsigned)iw < (unsigned)g.W) ? simg[c * hw + ih * g.W + iw] : 0u;
      if (++kw == g.KW) { kw = 0; if (++kh == g.KH) { kh = 0; ++c; } }
    }
    const long o = (b * ohw + m) * K + k0;
    *reinterpret_cast<uint4*>(hi + o) = make_uint4(__byte_perm(e[0], e[1], 0x5410), __byte_perm(e[2], e[3], 0x5410),
                                                   __byte_perm(e[4], e[5], 0x5410), __byte_perm(e[6], e[7], 0x5410));
    if (lo)
      *reinterpret_cast<uint4*>(lo + o) = make_uint4(__byte_perm(e[0], e[1], 0x7632), __byte_perm(e[2], e[3], 0x7632),
                                                     __byte_perm(e[4], e[5], 0x7632), __byte_perm(e[6], e[7], 0x7632));
  }
}

// colT (K, M): one thread = 8 consecutive m of one k  (M % 8 == 0)
template <typename T>
__global__ void im2col_bf16_t_kernel(riqn_conv_geom g, const T* __restrict__ in, bf16* __restrict__ hiT) {
  const int K = g.Cin * g.KH * g.KW;
  const long M = (long)g.B * g.OH * g.OW, M8 = M / 8;
  const long total = M8 * K;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const long m0 = (idx % M8) * 8;
    const int k = (int)(idx / M8);
    const int kw = k % g.KW, kh = (k / g.KW) % g.KH, c = k / (g.KW * g.KH);
    int ow = (int)(m0 % g.OW), oh = (int)((m0 / g.OW) % g.OH);
    long b = m0 / ((long)g.OW * g.OH);
    float x[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int ih = oh * g.stride + kh - g.pad, iw = ow * g.stride + kw - g.pad;
      x[t] = (ih >= 0 && ih < g.H && iw >= 0 && iw < g.W)
                 ? load_px<T>(&in[b * g.in_bstride + ((long)c * g.H + ih) * g.W + iw]) : 0.f;
      if (++ow == g.OW) { ow = 0; if (++oh == g.OH) { oh = 0; ++b; } }
    }
    uint4 h, l;
    pack8(x, h, l);
    *reinterpret_cast<uint4*>(hiT + (long)k * M + m0) = h;
  }
}

// dY = dout * (out > 0) from NCHW into the two bf16 operand layouts: dY (M, Cout) and dYT (Cout, M); the bias
// gradient (sum over b, p) is reduced per channel on the way.
__global__ void conv_dy_bf16_kernel(int B, int Cout, int ohw, const float* __restrict__ dout, const float* __restrict__ out,
                                    bf16* __restrict__ dY, bf16* __restrict__ dYT, float* __restrict__ dbias) {
  const int c = blockIdx.y;
  const long M = (long)B * ohw;
  float acc = 0.f;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (long)gridDim.x * blockDim.x) {
    const long b = i / ohw;
    const int p = (int)(i - b * ohw);
    const long src = (b * Cout + c) * ohw + p;
    const float v = out[src] > 0.f ? dout[src] : 0.f;
    acc += v;
    const bf16 h = __float2bfloat16_rn(v);
    if (dY) dY[i * Cout + c] = h;
    dYT[(long)c * M + i] = h;
  }
  acc = warp_sum(acc);
  __shared__ float red[32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(&dbias[c], v);
  }
}

// Tiled variant (Cout <= 64, Cout % 8 == 0): one block = 64 consecutive pixels x all channels.  NCHW reads and the dYT
// writes are coalesced along the pixels; the (M, Cout) image leaves through a shared tile as 16-byte row pieces.
__global__ void __launch_bounds__(256) conv_dy_tile_kernel(int B, int Cout, int ohw, const float* __restrict__ dout,
                                                           const float* __restrict__ out, bf16* __restrict__ dY,
                                                           bf16* __restrict__ dYT, float* __restrict__ dbias) {
  __shared__ __align__(16) unsigned short tile[64][66];
  __shared__ float bsum[64];
  const long M = (long)B * ohw;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < 64) bsum[threadIdx.x] = 0.f;
  __syncthreads();
  const long n_tiles = (M + 63) / 64;
  for (long tix = blockIdx.x; tix < n_tiles; tix += gridDim.x) {     // persistent: the bias partials stay in the block
    const long m0 = tix * 64;
    long src0[2];
    bool ok[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long m = m0 + lane + 32 * h;
      ok[h] = m < M;
      const long b = ok[h] ? m / ohw : 0;
      src0[h] = b * Cout * ohw + (ok[h] ? m - b * ohw : 0);       // + c * ohw
    }
    for (int c = warp; c < Cout; c += 8) {
      float acc = 0.f;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float v = 0.f;
        if (ok[h]) {
          const long src = src0[h] + (long)c * ohw;
          v = out[src] > 0.f ? dout[src] : 0.f;
        }
        const bf16 hb = __float2bfloat16_rn(v);
        if (ok[h]) dYT[(long)c * M + m0 + lane + 32 * h] = hb;
        tile[lane + 32 * h][c] = __bfloat16_as_ushort(hb);
        acc += v;
      }
      acc = warp_sum(acc);
      if (lane == 0) bsum[c] += acc;                               // channel c belongs to this warp only
    }
    __syncthreads();
    if (dY) {
      const int ppr = Cout >> 3;                                   // 16-byte pieces per row
      for (int idx = threadIdx.x; idx < 64 * ppr; idx += blockDim.x) {
        const int r = idx / ppr, pc = idx - r * ppr;
        if (m0 + r < M) {
          const uint32_t* w = reinterpret_cast<const uint32_t*>(&tile[r][pc * 8]);
          *reinterpret_cast<uint4*>(dY + (m0 + r) * Cout + pc * 8) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
    }
    __syncthreads();
  }
  if (threadIdx.x < Cout) atomicAdd(&dbias[threadIdx.x], bsum[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------------------------
// Strip convolution (forward without an im2col matrix).  With kernel edge k = t * stride, cut the (zero-padded) input
// into stride x stride blocks: block row r = (b, gy, gx) holds Kc = stride^2 * Cin values, and the im2col row of output
// (b, oy, ox) is the concatenation of the t x t blocks (oy + dy, ox + dx).  Laying the OUTPUTS on the same G x G block
// grid (G = OH + t - 1; only gy < OH, gx < OW are real) makes k-block (dy, dx) of an output tile the block rows
// m0 + dy*G + dx ... : a plain 2-D TMA tile of the block matrix at a row offset (gemm_tc.cu, TC_CONV).
// ---------------------------------------------------------------------------------------------------------------
// First layer: uint8 frames -> block matrix of raw pixel values (exact in bf16), within-block order (c, iy, ix).
__global__ void __launch_bounds__(256) s2d_u8_kernel(riqn_conv_geom g, int G, const uint8_t* __restrict__ in,
                                                     bf16* __restrict__ a_px) {
  extern __shared__ __align__(16) uint8_t img[];
  const int chw = g.Cin * g.H * g.W, s = g.stride, ss = s * s, Kc = ss * g.Cin, K8 = Kc / 8;
  const long b = blockIdx.x;
  const uint4* src = reinterpret_cast<const uint4*>(in + b * g.in_bstride);
  for (int i = threadIdx.x; i < chw / 16; i += blockDim.x) reinterpret_cast<uint4*>(img)[i] = src[i];
  __syncthreads();
  const bool fast = s == 4 && g.pad == 1 && (g.W & 3) == 0 && (G - 1) * 4 + 2 < g.W && (G - 1) * 4 + 2 < g.H;
  if (fast) {
    // item = (block r, channel c, row pair iy0 in {0, 2}): bytes 4*gx-1 .. 4*gx+2 of two image rows = byte 3 of word
    // gx-1 and bytes 0..2 of word gx; converted with the 2^23 trick (exact)
    const uint32_t* img32 = reinterpret_cast<const uint32_t*>(img);
    const int wpr = g.W >> 2;
    auto cvt2 = [](uint32_t w, uint32_t sa, uint32_t sb) -> uint32_t {
      const float fa = __uint_as_float(__byte_perm(w, 0x4B000000u, sa)) - 8388608.0f;
      const float fb = __uint_as_float(__byte_perm(w, 0x4B000000u, sb)) - 8388608.0f;
      return __byte_perm(__float_as_uint(fa), __float_as_uint(fb), 0x7632);
    };
    for (int item = threadIdx.x; item < G * G * K8; item += blockDim.x) {
      const int r = item / K8, q = item - r * K8;               // q = c * 2 + (iy0 / 2)
      const int gy = r / G, gx = r - gy * G, c = q >> 1, iy0 = (q & 1) * 2;
      uint32_t o[4];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int y = gy * 4 + iy0 + h - 1;
        uint32_t w0 = 0u, w1 = 0u;
        if (y >= 0) {
          const uint32_t* rowp = img32 + (c * g.H + y) * wpr + gx;
          w0 = gx > 0 ? rowp[-1] : 0u;
          w1 = rowp[0];
        }
        const uint32_t a = __byte_perm(w0, w1, 0x0043);          // bytes: w0.3, w1.0
        o[2 * h] = cvt2(a, 0x7650, 0x7651);
        o[2 * h + 1] = cvt2(w1, 0x7651, 0x7652);
      }
      *reinterpret_cast<uint4*>(a_px + (b * G * G + r) * Kc + q * 8) = make_uint4(o[0], o[1], o[2], o[3]);
    }
    return;
  }
  for (int item = threadIdx.x; item < G * G * K8; item += blockDim.x) {
    const int r = item / K8, k0 = (item - r * K8) * 8;
    const int gy = r / G, gx = r - gy * G;
    uint32_t e[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int k = k0 + t, c = k / ss, rem = k - c * ss, iy = rem / s, ix = rem - iy * s;
      const int y = gy * s + iy - g.pad, x = gx * s + ix - g.pad;
      e[t] = ((unsigned)y < (unsigned)g.H && (unsigned)x < (unsigned)g.W)
                 ? __float_as_uint((float)img[(c * g.H + y) * g.W + x]) >> 16 : 0u;
    }
    *reinterpret_cast<uint4*>(a_px + (b * G * G + r) * Kc + k0) =
        make_uint4(e[0] | (e[1] << 16), e[2] | (e[3] << 16), e[4] | (e[5] << 16), e[6] | (e[7] << 16));
  }
}

static inline int grid_for(long total) {
  long b = (total + 255) / 256;
  return (int)(b > 148L * 32 ? 148L * 32 : (b < 1 ? 1 : b));
}

}  // namespace riqn

using namespace riqn;

RIQN_API int riqn_conv_fwd(const riqn_conv_geom* g, const void* in, int in_is_u8, const float* w, const float* bias,
                           float* col, float* out, void* stream) {
  riqn::note_launches(2);
  cudaStream_t s = (cudaStream_t)stream;
  const long M = (long)g->B * g->OH * g->OW;
  const int K = g->Cin * g->KH * g->KW;
  if (in_is_u8) im2col_kernel<uint8_t><<<grid_for(M * K), 256, 0, s>>>(*g, (const uint8_t*)in, col);
  else im2col_kernel<float><<<grid_for(M * K), 256, 0, s>>>(*g, (const float*)in, col);
  RIQN_LAUNCH_CHECK();
  EpiArgs e;
  e.bias = bias;
  e.ohw = g->OH * g->OW;
  return gemm_f32((int)M, g->Cout, K, col, K, 1, w, K, 1, out, g->Cout, EPI_BIAS_RELU_NCHW, e, 1, s);
}

RIQN_API int riqn_im2col_f32(const riqn_conv_geom* g, const void* in, int in_is_u8, float* col, void* stream) {
  riqn::note_launches(1);
  cudaStream_t s = (cudaStream_t)stream;
  const long M = (long)g->B * g->OH * g->OW;
  const int K = g->Cin * g->KH * g->KW;
  if (in_is_u8) im2col_kernel<uint8_t><<<grid_for(M * K), 256, 0, s>>>(*g, (const uint8_t*)in, col);
  else im2col_kernel<float><<<grid_for(M * K), 256, 0, s>>>(*g, (const float*)in, col);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_conv_bwd(const riqn_conv_geom* g, const float* dout, const float* out, const float* col,
                           const float* w, float* dY, float* dcol, float* dw, float* dbias, float* din, void* stream) {
  riqn::note_launches(din ? 5 : 3);
  cudaStream_t s = (cudaStream_t)stream;
  const long M = (long)g->B * g->OH * g->OW;
  const int K = g->Cin * g->KH * g->KW;
  const int ohw = g->OH * g->OW;
  conv_dy_kernel<<<grid_for(M * g->Cout), 256, 0, s>>>(g->B, g->Cout, ohw, dout, out, dY);
  RIQN_LAUNCH_CHECK();
  int rc = colsum_atomic(M, g->Cout, dY, dbias, s);
  if (rc) return rc;
  // dW[c, k] += sum_m dY[m, c] * col[m, k]
  EpiArgs e;
  const int tiles = ((g->Cout + 127) / 128) * ((K + 127) / 128);
  int split = (2 * 148 + tiles - 1) / tiles;
  if ((long)split * 64 > M) split = (int)((M + 63) / 64);
  rc = gemm_f32(g->Cout, K, (int)M, dY, 1, g->Cout, col, 1, K, dw, K, EPI_ATOMIC, e, split, s);
  if (rc) return rc;
  if (din) {
    // dcol[m, k] = sum_c dY[m, c] * W[c, k]
    rc = gemm_f32((int)M, K, g->Cout, dY, g->Cout, 1, w, 1, K, dcol, K, EPI_STORE, e, 1, s);
    if (rc) return rc;
    rc = col2im(g, dcol, din, s);
    if (rc) return rc;
  }
  return 0;
}


// ---------------------------------------------------------------------------------------------------------------
// Tensor-core conv entry points (tcgen05 GEMM on bf16 hi/lo im2col operands)
// ---------------------------------------------------------------------------------------------------------------
RIQN_API int riqn_conv_fwd_tc(const riqn_conv_geom* g, const void* in, int in_is_u8, const void* w_hi, const void* w_lo,
                              const float* bias, void* col_hi, void* col_lo, void* colT_hi, float* out, void* stream) {
  riqn::note_launches(colT_hi ? 3 : 2);
  cudaStream_t s = (cudaStream_t)stream;
  const long M = (long)g->B * g->OH * g->OW;
  const int K = g->Cin * g->KH * g->KW;
  if (K % 8 || (colT_hi && M % 8)) return (int)cudaErrorInvalidValue;
  if (in_is_u8) im2col_bf16_u8_kernel<<<grid_for(M * K / 8), 256, 0, s>>>(*g, (const uint8_t*)in, (bf16*)col_hi, (bf16*)col_lo);
  else {
    const int chw = g->Cin * g->H * g->W;
    if (chw % 4 == 0 && g->in_bstride % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 && chw * 4 <= 96 * 1024) {
      static PerDeviceOnce attr_once;
      const int attr_dev = PerDeviceOnce::device();
      if (!attr_once.done[attr_dev]) {
        RIQN_CUDA(cudaFuncSetAttribute(im2col_f32_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
        attr_once.done[attr_dev] = true;
      }
      im2col_f32_staged_kernel<<<g->B, 256, (size_t)chw * 4, s>>>(*g, (const float*)in, (bf16*)col_hi, (bf16*)col_lo);
    } else {
      im2col_bf16_kernel<float><<<grid_for(M * K / 8), 256, 0, s>>>(*g, (const float*)in, (bf16*)col_hi, (bf16*)col_lo);
    }
  }
  RIQN_LAUNCH_CHECK();
  if (colT_hi) {
    if (in_is_u8) im2col_bf16_t_kernel<uint8_t><<<grid_for(M * K / 8), 256, 0, s>>>(*g, (const uint8_t*)in, (bf16*)colT_hi);
    else im2col_bf16_t_kernel<float><<<grid_for(M * K / 8), 256, 0, s>>>(*g, (const float*)in, (bf16*)colT_hi);
    RIQN_LAUNCH_CHECK();
  }
  TcExtra ex;
  ex.ohw = g->OH * g->OW;
  return gemm_bf16_tc((int)M, g->Cout, K, (const bf16*)col_hi, (const bf16*)col_lo, (const bf16*)w_hi,
                      col_lo ? (const bf16*)w_lo : nullptr, out, g->Cout, TC_BIAS_RELU_NCHW, bias, nullptr, nullptr, 1, s, &ex);
}

// First layer on raw uint8 pixels: A = pixel values (exact in bf16, no lo image), B = bf16 hi (+lo) of weight/255.
RIQN_API int riqn_conv_fwd_tc_u8(const riqn_conv_geom* g, const unsigned char* in, const void* ws_hi, const void* ws_lo,
                                 const float* bias, void* col_px, void* colT_px, float* out, int reuse_col, void* stream) {
  riqn::note_launches(reuse_col ? 1 : 2);
  cudaStream_t s = (cudaStream_t)stream;
  const long M = (long)g->B * g->OH * g->OW;
  const int K = g->Cin * g->KH * g->KW, chw = g->Cin * g->H * g->W, ohw = g->OH * g->OW;
  if (K % 8 || chw % 16 || g->in_bstride % 16 || (reinterpret_cast<uintptr_t>(in) & 15) || (colT_px && ohw % 8) || chw > 96 * 1024)
    return (int)cudaErrorInvalidValue;
  static PerDeviceOnce attr_once;
  const int attr_dev = PerDeviceOnce::device();
  if (!attr_once.done[attr_dev]) {
    RIQN_CUDA(cudaFuncSetAttribute(im2col_u8_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    attr_once.done[attr_dev] = true;
  }
  if (!reuse_col) {      // reuse_col: col_px already holds this input's im2col (another network's pass over it)
    im2col_u8_staged_kernel<<<dim3(g->B, 4), 256, chw, s>>>(*g, in, (bf16*)col_px, (bf16*)colT_px);
    RIQN_LAUNCH_CHECK();
  }
  TcExtra ex;
  ex.ohw = ohw;
  return gemm_bf16_tc((int)M, g->Cout, K, (const bf16*)col_px, nullptr, (const bf16*)ws_hi, (const bf16*)ws_lo, out, g->Cout,
                      TC_BIAS_RELU_NCHW, bias, nullptr, nullptr, 1, s, &ex);
}

// dY on the strip grid: row m' = (b, gy, gx) of dYg (B*G*G, Cout) bf16 holds dout * (out > 0) for real outputs
// (gy < OH, gx < OW) and zeros elsewhere; dbias accumulated.  One block = 64 grid rows x all channels (Cout <= 64).
__global__ void __launch_bounds__(256) conv_dy_grid_kernel(int B, int Cout, int OH, int OW, int G,
                                                           const float* __restrict__ dout, const float* __restrict__ out,
                                                           bf16* __restrict__ dYg, float* __restrict__ dbias) {
  __shared__ __align__(16) unsigned short tile[64][66];
  __shared__ float bsum[64];
  const long Mg = (long)B * G * G;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, ohw = OH * OW, gg = G * G;
  if (threadIdx.x < 64) bsum[threadIdx.x] = 0.f;
  __syncthreads();
  const long n_tiles = (Mg + 63) / 64;
  for (long tix = blockIdx.x; tix < n_tiles; tix += gridDim.x) {
    const long m0 = tix * 64;
    long src0[2];
    bool ok[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long m = m0 + lane + 32 * h;
      const long b = m / gg;
      const int rem = (int)(m - b * gg), gy = rem / G, gx = rem - gy * G;
      ok[h] = m < Mg && gy < OH && gx < OW;
      src0[h] = ok[h] ? b * Cout * ohw + gy * OW + gx : 0;          // + c * ohw
    }
    for (int c0 = warp; c0 < Cout; c0 += 32) {          // four channels (c0, +8, +16, +24) per pass: 16 loads in flight
      float o_[4][2], d_[4][2];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c = c0 + 8 * u;
          const bool on = ok[h] && c < Cout;
          const long src = src0[h] + (long)c * ohw;
          o_[u][h] = on ? __ldg(out + src) : 0.f;
          d_[u][h] = on ? __ldg(dout + src) : 0.f;
        }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int c = c0 + 8 * u;
        if (c < Cout) {
          float acc = 0.f;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float v = o_[u][h] > 0.f ? d_[u][h] : 0.f;
            tile[lane + 32 * h][c] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
            acc += v;
          }
          acc = warp_sum(acc);
          if (lane == 0) bsum[c] += acc;
        }
      }
    }
    __syncthreads();
    const int ppr = Cout >> 3;
    for (int idx = threadIdx.x; idx < 64 * ppr; idx += blockDim.x) {
      const int r = idx / ppr, pc = idx - r * ppr;
      if (m0 + r < Mg) {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(&tile[r][pc * 8]);
        *reinterpret_cast<uint4*>(dYg + (m0 + r) * Cout + pc * 8) = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
    __syncthreads();
  }
  if (threadIdx.x < Cout) atomicAdd(&dbias[threadIdx.x], bsum[threadIdx.x]);
}

// dw[c, perm[k']] += dwp[c, k']: the strip weight gradient back into the (Cout, Cin*KH*KW) parameter order
__global__ void unpermute_add_kernel(int Cout, int K, const float* __restrict__ dwp, const int* __restrict__ perm,
                                     float* __restrict__ dw) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= Cout * K) return;
  const int c = idx / K, kp = idx - c * K;
  dw[(long)c * K + perm[kp]] += dwp[idx];
}

// Weight image of the strip data gradient (TC_DGRAD operand B, (Cout, t*t*Kc) row-major, Kc = s*s*Cin):
//   wd[co, (dy*t + dx)*Kc + n] = w[co, c, s*dy + sy, s*dx + sx],   n = (sy, c, sx), sx fastest
// -- the column order in which the TC_DGRAD epilogue stores din.  w is the (Cout, Cin*KH*KW) bf16 weight.
__global__ void dgrad_weight_kernel(riqn_conv_geom g, int t, const bf16* __restrict__ w, bf16* __restrict__ wd) {
  const int s = g.stride, sc = s * g.Cin, Kc = s * sc, K = g.Cin * g.KH * g.KW;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= g.Cout * K) return;
  const int co = idx / K, q = idx - co * K;
  const int sft = q / Kc, n = q - sft * Kc, dy = sft / t, dx = sft - dy * t;
  const int sy = n / sc, r = n - sy * sc, c = r / s, sx = r - c * s;
  wd[idx] = w[(long)co * K + (c * g.KH + s * dy + sy) * g.KW + s * dx + sx];
}

static int strip_params(const riqn_conv_geom* g, int* t, int* G, int* kc) {
  if (g->KH != g->KW || g->stride < 1 || g->KH % g->stride) return 1;
  *t = g->KH / g->stride;
  *G = g->OH + *t - 1;
  const int Kc = g->stride * g->stride * g->Cin;
  if (g->OH != g->OW || Kc % 64 || g->OH != (g->H + 2 * g->pad - g->KH) / g->stride + 1) return 1;
  *kc = Kc / 64;
  return 0;
}

RIQN_API int riqn_s2d_u8(const riqn_conv_geom* g, const unsigned char* in, void* a_px, void* stream) {
  riqn::note_launches(1);
  int t, G, kc;
  const int chw = g->Cin * g->H * g->W;
  if (strip_params(g, &t, &G, &kc) || chw % 16 || g->in_bstride % 16 || (reinterpret_cast<uintptr_t>(in) & 15) ||
      chw > 96 * 1024)
    return (int)cudaErrorInvalidValue;
  static PerDeviceOnce attr_once;
  const int attr_dev = PerDeviceOnce::device();
  if (!attr_once.done[attr_dev]) {
    RIQN_CUDA(cudaFuncSetAttribute(s2d_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    attr_once.done[attr_dev] = true;
  }
  s2d_u8_kernel<<<g->B, 256, chw, (cudaStream_t)stream>>>(*g, G, in, (bf16*)a_px);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_conv_fwd_strip(const riqn_conv_geom* g, const void* a_hi, const void* a_lo, const void* w_hi,
                                 const void* w_lo, const float* bias, float* out, void* next_hi, void* next_lo,
                                 int next_stride, int next_grid, const void* w2_hi, const void* w2_lo, const float* bias2,
                                 int share_a, void* stream) {
  riqn::note_launches(1);
  int t, G, kc;
  if (strip_params(g, &t, &G, &kc) || g->Cout > 64 || (next_hi && (next_stride < 1 || next_grid < 1)))
    return (int)cudaErrorInvalidValue;
  TcExtra ex;
  if (w2_hi != nullptr) {           // two networks over one stacked batch: g->B counts BOTH halves
    const long rows = (long)g->B * G * G;
    if ((g->B & 1) || (rows / 2) % 128 || bias2 == nullptr || (w_lo != nullptr) != (w2_lo != nullptr)) return (int)cudaErrorInvalidValue;
    ex.grp_mt = (int)(rows / 2 / 128);
    ex.b2_hi = (const bf16*)w2_hi; ex.b2_lo = (const bf16*)w2_lo; ex.bias2 = bias2;
    if (share_a) { ex.a_wrap = 1; ex.a_rows = rows / 2; }
  }
  ex.strip_t = t; ex.strip_G = G; ex.strip_kc = kc;
  ex.cv_oh = g->OH; ex.cv_ow = g->OW;
  ex.nx_hi = (bf16*)next_hi; ex.nx_lo = (bf16*)next_lo; ex.nx_s = next_stride; ex.nx_G = next_grid;
  return gemm_bf16_tc(g->B * G * G, g->Cout, g->Cin * g->KH * g->KW, (const bf16*)a_hi, (const bf16*)a_lo, (const bf16*)w_hi,
                      (const bf16*)w_lo, out, g->Cout, TC_CONV, bias, nullptr, nullptr, 1, (cudaStream_t)stream, &ex);
}

// Backward of a strip convolution (bf16 operands, fp32 accumulate) without im2col matrices or transposes:
//   dYg (B*G*G, Cout) = dout * (out > 0) on the strip grid;   dbias += column sums
//   dW'[c, (shift, within)] = sum_m' dYg[m', c] * a_hi[m' + shift offset, within]   (MN-major operands, shifted rows)
//   dw[c, perm[k']] += wgrad_scale * dW'[c, k']
//   din = sum_shift dYg[m' - shift offset] * Wd_shift   (pad == 0 only; din may be NULL): the forward's shifted-row product
//        with negative shifts on the same block grid (TC_DGRAD), every din element written once -- no col2im scatter.
//        Wd is the bf16 weight in (shift, sy, c, sx) column order, built in the front of dwp_scratch before the weight
//        gradient needs that buffer.
RIQN_API int riqn_conv_bwd_strip(const riqn_conv_geom* g, const float* dout, const float* out, const void* a_hi,
                                 const void* w_hi, const int* perm, void* dYg, float* dwp_scratch, float* dw, float* dbias,
                                 float* din, float wgrad_scale, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  int t, G, kc;
  if (strip_params(g, &t, &G, &kc) || g->Cout > 64 || g->Cout % 8 || (din && g->pad != 0)) return (int)cudaErrorInvalidValue;
  // pad == 0: G*stride <= H; a remainder row / column (H - KH not a multiple of the stride) is read by no output
  const bool margin = din && (G * g->stride != g->H || G * g->stride != g->W);
  riqn::note_launches(din ? (margin ? 7 : 6) : 4);
  const long Mg = (long)g->B * G * G;
  const int K = g->Cin * g->KH * g->KW;
  const long tiles = (Mg + 63) / 64;
  conv_dy_grid_kernel<<<(unsigned)(tiles < 148 * 4 ? tiles : 148 * 4), 256, 0, s>>>(g->B, g->Cout, g->OH, g->OW, G, dout, out,
                                                                                (bf16*)dYg, dbias);
  RIQN_LAUNCH_CHECK();
  if (din) {
    bf16* wd = reinterpret_cast<bf16*>(dwp_scratch);      // Cout*K bf16 in a buffer of Cout*K floats
    dgrad_weight_kernel<<<(g->Cout * K + 255) / 256, 256, 0, s>>>(*g, t, (const bf16*)w_hi, wd);
    RIQN_LAUNCH_CHECK();
    if (margin) RIQN_CUDA(cudaMemsetAsync(din, 0, sizeof(float) * (size_t)g->B * g->Cin * g->H * g->W, s));
    TcExtra dg;
    dg.strip_t = t; dg.strip_G = G; dg.dg_cout = g->Cout;
    dg.ci_h = g->H; dg.ci_w = g->W; dg.ci_cin = g->Cin; dg.ci_stride = g->stride;
    const int rc = gemm_bf16_tc((int)Mg, kc * 64, t * t * 64, (const bf16*)dYg, nullptr, wd, nullptr, din, 0, TC_DGRAD,
                                nullptr, nullptr, nullptr, 1, s, &dg);
    if (rc) return rc;
  }
  RIQN_CUDA(cudaMemsetAsync(dwp_scratch, 0, sizeof(float) * g->Cout * K, s));
  TcExtra ex;
  ex.mn_major = 3;
  ex.wg_t = t; ex.wg_G = G; ex.wg_kc = kc;
  ex.alpha = wgrad_scale;
  const int n_tiles = (K + 255) / 256;
  const int split = tc_pick_split(n_tiles, (Mg + 63) / 64);
  int rc = gemm_bf16_tc(g->Cout, K, (int)Mg, (const bf16*)dYg, nullptr, (const bf16*)a_hi, nullptr, dwp_scratch, K, TC_ATOMIC,
                        nullptr, nullptr, nullptr, split, s, &ex);
  if (rc) return rc;
  unpermute_add_kernel<<<(g->Cout * K + 255) / 256, 256, 0, s>>>(g->Cout, K, dwp_scratch, perm, dw);
  RIQN_LAUNCH_CHECK();
  return 0;
}

// bf16 transposed im2col (K, M) alone -- the wgrad operand of riqn_conv_bwd_tc when the forward ran as a strip
// convolution.  in_is_u8: raw pixel VALUES are written (pass wgrad_scale = 1/255 to riqn_conv_bwd_tc).
RIQN_API int riqn_im2col_bf16_t(const riqn_conv_geom* g, const void* in, int in_is_u8, void* colT_hi, void* stream) {
  riqn::note_launches(1);
  cudaStream_t s = (cudaStream_t)stream;
  const long M = (long)g->B * g->OH * g->OW;
  const int K = g->Cin * g->KH * g->KW, chw = g->Cin * g->H * g->W, ohw = g->OH * g->OW;
  if (K % 8 || M % 8) return (int)cudaErrorInvalidValue;
  if (in_is_u8) {
    if (chw % 16 || g->in_bstride % 16 || (reinterpret_cast<uintptr_t>(in) & 15) || ohw % 8 || chw > 96 * 1024)
      return (int)cudaErrorInvalidValue;
    static PerDeviceOnce attr_once;
    const int attr_dev = PerDeviceOnce::device();
    if (!attr_once.done[attr_dev]) {
      RIQN_CUDA(cudaFuncSetAttribute(im2col_u8_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
      attr_once.done[attr_dev] = true;
    }
    im2col_u8_staged_kernel<<<dim3(g->B, 4), 256, chw, s>>>(*g, (const unsigned char*)in, nullptr, (bf16*)colT_hi);
  } else {
    im2col_bf16_t_kernel<float><<<grid_for(M * K / 8), 256, 0, s>>>(*g, (const float*)in, (bf16*)colT_hi);
  }
  return (int)cudaGetLastError();
}

RIQN_API int riqn_conv_bwd_tc(const riqn_conv_geom* g, const float* dout, const float* out, const void* colT_hi,
                              const void* wT_hi, void* dY_hi, void* dYT_hi, float* dcol, float* dw, float* dbias, float* din,
                              float wgrad_scale, void* stream) {
  riqn::note_launches(din ? 4 : 2);
  cudaStream_t s = (cudaStream_t)stream;
  const long M = (long)g->B * g->OH * g->OW;
  const int K = g->Cin * g->KH * g->KW;
  const int ohw = g->OH * g->OW;
  if (M % 8 || g->Cout % 8) return (int)cudaErrorInvalidValue;
  if (g->Cout <= 64) {
    const long tiles = (M + 63) / 64;
    conv_dy_tile_kernel<<<(unsigned)(tiles < 148 * 4 ? tiles : 148 * 4), 256, 0, s>>>(g->B, g->Cout, ohw, dout, out,
                                                                 din ? (bf16*)dY_hi : nullptr, (bf16*)dYT_hi, dbias);
  } else {
    dim3 grid((unsigned)((M + 256 * 8 - 1) / (256 * 8)), g->Cout);
    conv_dy_bf16_kernel<<<grid, 256, 0, s>>>(g->B, g->Cout, ohw, dout, out, din ? (bf16*)dY_hi : nullptr, (bf16*)dYT_hi, dbias);
  }
  RIQN_LAUNCH_CHECK();
  // dW[c, k] += sum_m dY[m, c] * col[m, k]      (K' = M is long: split it over every SM)
  const int n_tiles = (K + 255) / 256;
  int split = (148 + n_tiles - 1) / n_tiles;
  TcExtra ex;
  ex.alpha = wgrad_scale;          // 1/255 when colT holds raw pixel values
  int rc = gemm_bf16_tc(g->Cout, K, (int)M, (const bf16*)dYT_hi, nullptr, (const bf16*)colT_hi, nullptr, dw, K, TC_ATOMIC,
                        nullptr, nullptr, nullptr, split, s, &ex);
  if (rc) return rc;
  if (din) {
    // dcol[m, k] = sum_c dY[m, c] * W[c, k]
    if (g->pad == 0) {
      // fused col2im: the accumulators are added straight into din (never materialising dcol)
      RIQN_CUDA(cudaMemsetAsync(din, 0, sizeof(float) * (size_t)g->B * g->Cin * g->H * g->W, s));
      TcExtra ci;
      ci.ohw = ohw;
      ci.ci_h = g->H; ci.ci_w = g->W; ci.ci_cin = g->Cin; ci.ci_kh = g->KH; ci.ci_kw = g->KW;
      ci.ci_stride = g->stride; ci.ci_ow = g->OW;
      rc = gemm_bf16_tc((int)M, K, g->Cout, (const bf16*)dY_hi, nullptr, (const bf16*)wT_hi, nullptr, din, K, TC_COL2IM,
                        nullptr, nullptr, nullptr, 1, s, &ci);
      if (rc) return rc;
    } else {
      rc = gemm_bf16_tc((int)M, K, g->Cout, (const bf16*)dY_hi, nullptr, (const bf16*)wT_hi, nullptr, dcol, K, TC_STORE,
                        nullptr, nullptr, nullptr, 1, s, nullptr);
      if (rc) return rc;
      rc = col2im(g, dcol, din, s);
      if (rc) return rc;
    }
  }
  return 0;
}
