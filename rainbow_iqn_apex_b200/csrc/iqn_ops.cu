// IQN head of the DQN and the quantile-Huber loss (reference rainbowiqn/model.py:9-53,130-157 and
// rainbowiqn/compute_loss_iqn.py:216-358) as CUDA ops behind the C-ABI in include/riqn_b200.h.
//
// Row conventions: the reference tiles rows quantile-major, r = q*B + b (model.py:149; compute_loss_iqn.py:238-310);
// tau, q and dtheta cross the C-ABI in that order.  INTERNALLY (cos, x, h, dh, dz) rows are sample-major,
// r' = b*Nq + q, so that the 32 lanes of a warp belong to one sample: the Hadamard operand feat[b,:] is then a
// warp-broadcast load and the reduction over a sample's quantiles is contiguous.
#include "common.cuh"
#include "gemm.h"
#include "../../include/riqn_b200.h"

namespace riqn {
int colsum_atomic(long M, int N, const float* X, float* out, cudaStream_t s);

// ------------------------------------------------------------------------------------------------
// RNG fills
// ------------------------------------------------------------------------------------------------
__global__ void fill_uniform_kernel(long n, uint64_t seed, uint64_t stream, float* __restrict__ out,
                                    const riqn_dyn_state* __restrict__ dyn) {
  if (dyn) stream += dyn->rng_offset;
  const long i4 = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 * 4 >= n) return;
  const uint4 r = Philox::draw(seed, stream, (uint64_t)i4);
  const float v[4] = {Philox::u01(r.x), Philox::u01(r.y), Philox::u01(r.z), Philox::u01(r.w)};
  for (int j = 0; j < 4; ++j)
    if (i4 * 4 + j < n) out[i4 * 4 + j] = v[j];
}

// f(x) = sign(x) sqrt|x| of x ~ N(0,1)            (NoisyLinear._scale_noise, model.py:32-37)
__global__ void fill_scaled_normal_kernel(long n, uint64_t seed, uint64_t stream, float* __restrict__ out,
                                          const riqn_dyn_state* __restrict__ dyn) {
  if (dyn) stream += dyn->rng_offset;
  const long i4 = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 * 4 >= n) return;
  const uint4 r = Philox::draw(seed, stream, (uint64_t)i4);
  const float u0 = Philox::u01(r.x), u1 = Philox::u01(r.y), u2 = Philox::u01(r.z), u3 = Philox::u01(r.w);
  const float ra = sqrtf(-2.f * logf(u0)), rb = sqrtf(-2.f * logf(u2));
  float s0, c0, s1, c1;
  sincospif(2.f * u1, &s0, &c0);
  sincospif(2.f * u3, &s1, &c1);
  const float z[4] = {ra * c0, ra * s0, rb * c1, rb * s1};
  for (int j = 0; j < 4; ++j)
    if (i4 * 4 + j < n) out[i4 * 4 + j] = copysignf(sqrtf(fabsf(z[j])), z[j]);
}

// ------------------------------------------------------------------------------------------------
// Quantile embedding input: cos(fl(fl(i) * fl(pi)) * tau), i = 1..E          (model.py:136-144)
// ------------------------------------------------------------------------------------------------
__global__ void cos_embed_kernel(int B, int Nq, int E, const float* __restrict__ tau, float* __restrict__ cosv) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)B * Nq * E) return;
  const int i = (int)(idx % E) + 1;
  const long r = idx / E;                                   // sample-major row b*Nq + q
  const int b = (int)(r / Nq), q = (int)(r - (long)b * Nq);
  const float ipi = __fmul_rn((float)i, 3.14159274101257324f);
  cosv[idx] = cosf(__fmul_rn(ipi, tau[(long)q * B + b]));   // tau arrives quantile-major
}

// Same values as bf16 (hi, lo) operand images for the tensor-core embedding product, plus the transposed hi image
// (E, R) the iqn_fc weight-gradient product consumes.
__global__ void cos_embed_bf16_kernel(int B, int Nq, int E, const float* __restrict__ tau, __nv_bfloat16* __restrict__ hi,
                                      __nv_bfloat16* __restrict__ lo, __nv_bfloat16* __restrict__ hiT) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long R = (long)B * Nq;
  if (idx >= R * E) return;
  const int i = (int)(idx % E) + 1;
  const long r = idx / E;                                   // sample-major row b*Nq + q
  const int b = (int)(r / Nq), q = (int)(r - (long)b * Nq);
  const float ipi = __fmul_rn((float)i, 3.14159274101257324f);
  const float c = cosf(__fmul_rn(ipi, tau[(long)q * B + b]));
  const __nv_bfloat16 h = __float2bfloat16_rn(c);
  hi[idx] = h;
  if (lo) lo[idx] = __float2bfloat16_rn(c - __bfloat162float(h));
  if (hiT) hiT[(long)(i - 1) * R + r] = h;
}

// Backward through x = feat[b] (.) phi[r] on bf16 operand images:
//   x = x_hi (+ x_lo);  dpre = dX * feat * 1{x>0}  -> dpre (R, F) bf16 row-major (MN-major operand of the dW_e product)
//   dfeat[b,f] = (sum_q dX * x) / feat ;  dbe[f] += sum_r dpre
// Rows are sample-major, so one block = one sample x 32 features walks that sample's Nq contiguous rows.
__global__ void embed_bwd_tile_kernel(int B, int Nq, int F, const __nv_bfloat16* __restrict__ x_hi,
                                      const __nv_bfloat16* __restrict__ x_lo, const float* __restrict__ feat,
                                      const float* __restrict__ dX, const __nv_bfloat16* __restrict__ dXb,
                                      __nv_bfloat16* __restrict__ dpre, float* __restrict__ dfeat,
                                      float* __restrict__ dbe) {
  __shared__ float red[2][8][32];
  const int f0 = blockIdx.x * 32, b = blockIdx.y;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  const int f = f0 + tx;
  const float ft = f < F ? feat[(long)b * F + f] : 0.f;
  float facc = 0.f, bacc = 0.f;
  for (int q = ty; q < Nq; q += 8) {
    if (f < F) {
      const long o = ((long)b * Nq + q) * F + f;
      float x = __bfloat162float(x_hi[o]);
      if (x_lo) x += __bfloat162float(x_lo[o]);
      const float dx = dXb ? __bfloat162float(dXb[o]) : dX[o];
      facc = fmaf(dx, x, facc);
      const float dp = x > 0.f ? dx * ft : 0.f;
      bacc += dp;
      dpre[o] = __float2bfloat16_rn(dp);
    }
  }
  red[0][ty][tx] = facc;
  red[1][ty][tx] = bacc;
  __syncthreads();
  if (ty == 0 && f < F) {
    float fs = 0.f, bs = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { fs += red[0][j][tx]; bs += red[1][j][tx]; }
    dfeat[(long)b * F + f] = ft > 0.f ? fs / ft : 0.f;
    atomicAdd(&dbe[f], bs);
  }
}

// Wide variant (Nq even): one block = one sample x 128 features; lane owns 4 consecutive features (16-byte dX loads,
// 8-byte x loads, 8-byte dpre stores), warp w owns rows q = 2w, 2w+1, 2w+16, ... so that all of a thread's loads are in
// flight together.
template <bool DXB, bool XLO>
__global__ void __launch_bounds__(256) embed_bwd_wide_kernel(int B, int Nq, int F, const __nv_bfloat16* __restrict__ x_hi,
                                                             const __nv_bfloat16* __restrict__ x_lo,
                                                             const float* __restrict__ feat, const float* __restrict__ dX,
                                                             const __nv_bfloat16* __restrict__ dXb,
                                                             __nv_bfloat16* __restrict__ dpre, float* __restrict__ dfeat,
                                                             float* __restrict__ dbe) {
  __shared__ float red[2][8][128];
  const int f0 = blockIdx.x * 128, b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long R = (long)B * Nq;
  const int fl = 4 * lane, f = f0 + fl;                 // F % 4 == 0 is checked by the host
  const bool f_ok = f < F;
  float4 ft = make_float4(0.f, 0.f, 0.f, 0.f);
  if (f_ok) ft = *reinterpret_cast<const float4*>(feat + (long)b * F + f);
  float facc[4] = {0.f, 0.f, 0.f, 0.f}, bacc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int q0 = 0; q0 < Nq; q0 += 64) {
    // rows handled by this thread in this pass: q0 + 2*(warp + 8*i) + {0, 1}, i < 4
    float4 dx[8];
    uint2 xh[8], xl[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int q = q0 + 2 * (warp + 8 * (i >> 1)) + (i & 1);
      dx[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      xh[i] = make_uint2(0u, 0u);
      xl[i] = make_uint2(0u, 0u);
      if (q < Nq && f_ok) {
        const long o = ((long)b * Nq + q) * F + f;
        if (DXB) {                                             // bf16 dX: 8-byte loads
          const uint2 d2 = __ldg(reinterpret_cast<const uint2*>(dXb + o));
          dx[i] = make_float4(__uint_as_float(d2.x << 16), __uint_as_float(d2.x & 0xffff0000u), __uint_as_float(d2.y << 16),
                              __uint_as_float(d2.y & 0xffff0000u));
        } else {
          dx[i] = __ldg(reinterpret_cast<const float4*>(dX + o));
        }
        xh[i] = __ldg(reinterpret_cast<const uint2*>(x_hi + o));
        if (XLO) xl[i] = __ldg(reinterpret_cast<const uint2*>(x_lo + o));
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int q = q0 + 2 * (warp + 8 * (i >> 1)) + (i & 1);
      const float x[4] = {__uint_as_float(xh[i].x << 16) + __uint_as_float(xl[i].x << 16),
                          __uint_as_float(xh[i].x & 0xffff0000u) + __uint_as_float(xl[i].x & 0xffff0000u),
                          __uint_as_float(xh[i].y << 16) + __uint_as_float(xl[i].y << 16),
                          __uint_as_float(xh[i].y & 0xffff0000u) + __uint_as_float(xl[i].y & 0xffff0000u)};
      const float d[4] = {dx[i].x, dx[i].y, dx[i].z, dx[i].w};
      const float fv[4] = {ft.x, ft.y, ft.z, ft.w};
      float dp[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        facc[j] = fmaf(d[j], x[j], facc[j]);
        dp[j] = x[j] > 0.f ? d[j] * fv[j] : 0.f;
        bacc[j] += dp[j];
      }
      if (q < Nq && f_ok) {                                  // dpre (R, F) row-major: 8 bytes per lane, 256 per warp
        const __nv_bfloat162 p01 = __floats2bfloat162_rn(dp[0], dp[1]), p23 = __floats2bfloat162_rn(dp[2], dp[3]);
        *reinterpret_cast<uint2*>(dpre + ((long)b * Nq + q) * F + f) =
            make_uint2(*reinterpret_cast<const uint32_t*>(&p01), *reinterpret_cast<const uint32_t*>(&p23));
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    red[0][warp][fl + j] = facc[j];
    red[1][warp][fl + j] = bacc[j];
  }
  __syncthreads();
  if (threadIdx.x < 128 && f0 + threadIdx.x < F) {
    const int t = threadIdx.x;
    float fs = 0.f, bs = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { fs += red[0][j][t]; bs += red[1][j][t]; }
    const float fv = feat[(long)b * F + f0 + t];
    dfeat[(long)b * F + f0 + t] = fv > 0.f ? fs / fv : 0.f;
    atomicAdd(&dbe[f0 + t], bs);
  }
}

// bf16-dX variant with 16-byte accesses throughout: lane owns 8 consecutive features (one block = one sample x 256
// features), warp w owns rows q = w, w+8, ...; all of a thread's loads of a 64-row pass are in flight together.
template <bool XLO>
__global__ void __launch_bounds__(256) embed_bwd_wide8_kernel(int B, int Nq, int F, const __nv_bfloat16* __restrict__ x_hi,
                                                              const __nv_bfloat16* __restrict__ x_lo,
                                                              const float* __restrict__ feat,
                                                              const __nv_bfloat16* __restrict__ dXb,
                                                              __nv_bfloat16* __restrict__ dpre, float* __restrict__ dfeat,
                                                              float* __restrict__ dbe) {
  __shared__ float red[2][8][256];
  const int f0 = blockIdx.x * 256, b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int fl = 8 * lane, f = f0 + fl;                 // F % 8 == 0 is checked by the host
  const bool f_ok = f < F;
  float fv[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) fv[j] = 0.f;
  if (f_ok) {
    const float4 a = *reinterpret_cast<const float4*>(feat + (long)b * F + f);
    const float4 c = *reinterpret_cast<const float4*>(feat + (long)b * F + f + 4);
    fv[0] = a.x; fv[1] = a.y; fv[2] = a.z; fv[3] = a.w; fv[4] = c.x; fv[5] = c.y; fv[6] = c.z; fv[7] = c.w;
  }
  float facc[8], bacc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { facc[j] = 0.f; bacc[j] = 0.f; }
  auto lo16 = [](uint32_t w) { return __uint_as_float(w << 16); };
  auto hi16 = [](uint32_t w) { return __uint_as_float(w & 0xffff0000u); };
  for (int q0 = 0; q0 < Nq; q0 += 64) {
    uint4 dx[8], xh[8], xl[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int q = q0 + warp + 8 * i;
      dx[i] = make_uint4(0u, 0u, 0u, 0u);
      xh[i] = make_uint4(0u, 0u, 0u, 0u);
      xl[i] = make_uint4(0u, 0u, 0u, 0u);
      if (q < Nq && f_ok) {
        const long o = ((long)b * Nq + q) * F + f;
        dx[i] = __ldg(reinterpret_cast<const uint4*>(dXb + o));
        xh[i] = __ldg(reinterpret_cast<const uint4*>(x_hi + o));
        if (XLO) xl[i] = __ldg(reinterpret_cast<const uint4*>(x_lo + o));
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int q = q0 + warp + 8 * i;
      const uint32_t dw[4] = {dx[i].x, dx[i].y, dx[i].z, dx[i].w}, hw[4] = {xh[i].x, xh[i].y, xh[i].z, xh[i].w},
                     lw[4] = {xl[i].x, xl[i].y, xl[i].z, xl[i].w};
      uint32_t ow[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float x0 = lo16(hw[k]) + lo16(lw[k]), x1 = hi16(hw[k]) + hi16(lw[k]);
        const float d0 = lo16(dw[k]), d1 = hi16(dw[k]);
        facc[2 * k] = fmaf(d0, x0, facc[2 * k]);
        facc[2 * k + 1] = fmaf(d1, x1, facc[2 * k + 1]);
        const float p0 = x0 > 0.f ? d0 * fv[2 * k] : 0.f, p1 = x1 > 0.f ? d1 * fv[2 * k + 1] : 0.f;
        bacc[2 * k] += p0;
        bacc[2 * k + 1] += p1;
        const __nv_bfloat162 pp = __floats2bfloat162_rn(p0, p1);
        ow[k] = *reinterpret_cast<const uint32_t*>(&pp);
      }
      if (q < Nq && f_ok)
        *reinterpret_cast<uint4*>(dpre + ((long)b * Nq + q) * F + f) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    red[0][warp][fl + j] = facc[j];
    red[1][warp][fl + j] = bacc[j];
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (f0 + t < F) {
    float fs = 0.f, bs = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) { fs += red[0][j][t]; bs += red[1][j][t]; }
    const float ftv = feat[(long)b * F + f0 + t];
    dfeat[(long)b * F + f0 + t] = ftv > 0.f ? fs / ftv : 0.f;
    atomicAdd(&dbe[f0 + t], bs);
  }
}

// ------------------------------------------------------------------------------------------------
// NoisyLinear: (optional) eps_w = eps_out (x) eps_in, then W_eff = mu + sigma*eps_w, b_eff likewise
// (model.py:39-53).  training == 0 gives the eval-mode weights (mu only).
// ------------------------------------------------------------------------------------------------
__global__ void noisy_compose_kernel(int out_f, int in_f, const float* __restrict__ mu, const float* __restrict__ sigma,
                                     float* __restrict__ eps_w, const float* __restrict__ eps_in,
                                     const float* __restrict__ eps_out, const float* __restrict__ bmu,
                                     const float* __restrict__ bsigma, float* __restrict__ beps,
                                     float* __restrict__ w_eff, float* __restrict__ b_eff, int training) {
  const long total = (long)out_f * in_f;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int o = (int)(idx / in_f), i = (int)(idx % in_f);
    float e;
    if (eps_in) {
      e = __fmul_rn(eps_out[o], eps_in[i]);
      eps_w[idx] = e;
    } else {
      e = eps_w[idx];
    }
    w_eff[idx] = training ? __fadd_rn(mu[idx], __fmul_rn(sigma[idx], e)) : mu[idx];
    if (i == 0) {
      float eb;
      if (eps_in) {
        eb = eps_out[o];
        beps[o] = eb;
      } else {
        eb = beps[o];
      }
      b_eff[o] = training ? __fadd_rn(bmu[o], __fmul_rn(bsigma[o], eb)) : bmu[o];
    }
  }
}

// Network-wide variants: the (<= 8) layers of a network travel by value in the launch parameters.
struct NoisyNet {
  riqn_noisy_layer l[8];
  int n;
  int blk_end[16];     // exclusive prefix of blocks per segment (fill: 2 per layer) / per layer (compose)
};

__global__ void noisy_fill_net_kernel(NoisyNet net, uint64_t seed, const riqn_dyn_state* __restrict__ dyn) {
  int seg = 0;
  while (seg < 2 * net.n - 1 && (int)blockIdx.x >= net.blk_end[seg]) ++seg;
  const riqn_noisy_layer& L = net.l[seg >> 1];
  const bool is_out = seg & 1;
  const long n = is_out ? L.out_features : L.in_features;
  float* out = is_out ? L.eps_out : L.eps_in;
  uint64_t stream = is_out ? L.stream_out : L.stream_in;
  if (dyn) stream += dyn->rng_offset;
  const long i4 = (long)(blockIdx.x - (seg ? net.blk_end[seg - 1] : 0)) * blockDim.x + threadIdx.x;
  if (i4 * 4 >= n) return;
  const uint4 r = Philox::draw(seed, stream, (uint64_t)i4);                 // identical to fill_scaled_normal_kernel
  const float u0 = Philox::u01(r.x), u1 = Philox::u01(r.y), u2 = Philox::u01(r.z), u3 = Philox::u01(r.w);
  const float ra = sqrtf(-2.f * logf(u0)), rb = sqrtf(-2.f * logf(u2));
  float s0, c0, s1, c1;
  sincospif(2.f * u1, &s0, &c0);
  sincospif(2.f * u3, &s1, &c1);
  const float z[4] = {ra * c0, ra * s0, rb * c1, rb * s1};
  for (int j = 0; j < 4; ++j)
    if (i4 * 4 + j < n) out[i4 * 4 + j] = copysignf(sqrtf(fabsf(z[j])), z[j]);
}

// one thread = 4 consecutive inputs of one output row (16-byte accesses); block ranges per layer from blk_end
__global__ void noisy_compose_net_kernel(NoisyNet net, int training) {
  int li = 0;
  while (li < net.n - 1 && (int)blockIdx.x >= net.blk_end[li]) ++li;
  const riqn_noisy_layer& L = net.l[li];
  const int in4 = L.in_features >> 2;
  const int total = L.out_features * in4;
  const int idx = (blockIdx.x - (li ? net.blk_end[li - 1] : 0)) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int o = idx / in4, i = (idx - o * in4) * 4;
  const float eo = L.eps_out[o];
  const float4 ei = *reinterpret_cast<const float4*>(L.eps_in + i);
  const long off = (long)o * L.in_features + i;
  const float4 e = make_float4(__fmul_rn(eo, ei.x), __fmul_rn(eo, ei.y), __fmul_rn(eo, ei.z), __fmul_rn(eo, ei.w));
  *reinterpret_cast<float4*>(L.weight_epsilon + off) = e;
  const float4 mu = *reinterpret_cast<const float4*>(L.weight_mu + off);
  float4 w = mu;
  if (training) {
    const float4 sg = *reinterpret_cast<const float4*>(L.weight_sigma + off);
    w = make_float4(__fadd_rn(mu.x, __fmul_rn(sg.x, e.x)), __fadd_rn(mu.y, __fmul_rn(sg.y, e.y)),
                    __fadd_rn(mu.z, __fmul_rn(sg.z, e.z)), __fadd_rn(mu.w, __fmul_rn(sg.w, e.w)));
  }
  *reinterpret_cast<float4*>(L.w_eff + off) = w;
  if (L.w_hi != nullptr && L.w_fp16) {   // fp16(w) for the single-pass head forward, bf16(w) (optional) for the data gradient
    const __half2 h01 = __floats2half2_rn(w.x, w.y), h23 = __floats2half2_rn(w.z, w.w);
    *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(L.w_hi) + off) =
        make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
    if (L.w_lo != nullptr) {
      const __nv_bfloat162 b01 = __floats2bfloat162_rn(w.x, w.y), b23 = __floats2bfloat162_rn(w.z, w.w);
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(L.w_lo) + off) =
          make_uint2(*reinterpret_cast<const uint32_t*>(&b01), *reinterpret_cast<const uint32_t*>(&b23));
    }
  } else if (L.w_hi != nullptr) {    // bf16 operand images written here instead of by a separate split pass
    const __nv_bfloat162 h01 = __floats2bfloat162_rn(w.x, w.y), h23 = __floats2bfloat162_rn(w.z, w.w);
    const uint32_t u01 = *reinterpret_cast<const uint32_t*>(&h01), u23 = *reinterpret_cast<const uint32_t*>(&h23);
    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(L.w_hi) + off) = make_uint2(u01, u23);
    if (L.w_lo != nullptr) {
      const __nv_bfloat162 l01 = __floats2bfloat162_rn(w.x - __uint_as_float(u01 << 16), w.y - __uint_as_float(u01 & 0xffff0000u));
      const __nv_bfloat162 l23 = __floats2bfloat162_rn(w.z - __uint_as_float(u23 << 16), w.w - __uint_as_float(u23 & 0xffff0000u));
      *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(L.w_lo) + off) =
          make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
    }
  }
  if (i == 0) {
    L.bias_epsilon[o] = eo;
    L.b_eff[o] = training ? __fadd_rn(L.bias_mu[o], __fmul_rn(L.bias_sigma[o], eo)) : L.bias_mu[o];
  }
}

// ------------------------------------------------------------------------------------------------
// z-layers + dueling: q[r,a] = v + a_a - mean_a(a)                           (model.py:153-156)
//   H (R, 2*hid): [:, :hid] value stream hidden, [:, hid:] advantage stream hidden (post-ReLU)
//   Wz (1+A, hid): row 0 = z_v effective weight, rows 1.. = z_a ; bz (1+A)
// One warp per row.
// ------------------------------------------------------------------------------------------------
template <int HID>
__global__ void z_dueling_fwd_kernel(long R, int B, int A, const float* __restrict__ H, const float* __restrict__ Wz,
                                     const float* __restrict__ bz, float* __restrict__ q) {
  extern __shared__ float sW[];  // (1+A) * HID
  for (int i = threadIdx.x; i < (1 + A) * HID; i += blockDim.x) sW[i] = Wz[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  constexpr int T = HID / 32;
  for (long r = (long)blockIdx.x * wpb + warp; r < R; r += (long)gridDim.x * wpb) {
    const float* h = H + r * (2 * HID);
    float hv[T], ha[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
      hv[t] = h[lane + 32 * t];
      ha[t] = h[HID + lane + 32 * t];
    }
    float v = 0.f;
#pragma unroll
    for (int t = 0; t < T; ++t) v = fmaf(hv[t], sW[lane + 32 * t], v);
    v = warp_sum(v) + bz[0];
    float mine = 0.f, asum = 0.f;
    for (int k = 0; k < A; ++k) {
      float a = 0.f;
      const float* wk = sW + (1 + k) * HID;
#pragma unroll
      for (int t = 0; t < T; ++t) a = fmaf(ha[t], wk[lane + 32 * t], a);
      a = warp_sum(a) + bz[1 + k];
      asum += a;
      if (lane == k) mine = a;
    }
    const int Nq = (int)(R / B);
    const long b = r / Nq, qi = r - b * Nq;                 // sample-major row -> quantile-major output row
    if (lane < A) q[(qi * B + b) * A + lane] = v + mine - asum / (float)A;
  }
}

// Four rows per warp: every weight fetched from shared memory (16-byte reads) is used for four rows, all 32 row loads
// of a thread are in flight together, and the four dot products of one output are reduced with 6 shuffles (a
// transpose-reduce over lane bits 4 and 3, then a butterfly over bits 2..0): lane l ends up with the sums of row
// rr(l) = 2*bit3(l) + bit4(l), and the 8 lanes of a row share out the A advantages.
// The row registers hx[4][HID/128] are 16*HID/128 floats: up to 512 they fit two blocks per SM (128-register cap); wider
// layers run one block per SM so that nothing spills.
template <int HID>
constexpr int zd_fwd4_min_blocks() { return HID <= 512 ? 2 : 1; }

template <int HID>
__global__ void __launch_bounds__(256, zd_fwd4_min_blocks<HID>()) z_dueling_fwd4_kernel(long R, int B, int A,
                                                                                        const float* __restrict__ H,
                                                                                        const float* __restrict__ Wz,
                                                                                        const float* __restrict__ bz,
                                                                                        float* __restrict__ q) {
  extern __shared__ float sW[];  // (1+A) * HID
  for (int i = threadIdx.x; i < (1 + A) * HID / 4; i += blockDim.x)
    reinterpret_cast<float4*>(sW)[i] = reinterpret_cast<const float4*>(Wz)[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  constexpr int T = HID / 128;
  const int Nq = (int)(R / B);
  const int my_rr = ((lane >> 3) & 1) * 2 + ((lane >> 4) & 1), my_j = lane & 7;
  // one output: 4 rows x (T float4) against weight row k; returns the sum of row rr(lane) on every lane
  auto dot4 = [&](const float4 (&hx)[4][T], int k) -> float {
    const float4* wk = reinterpret_cast<const float4*>(sW + k * HID);
    float p[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const float4 w = wk[lane + 32 * t];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const float4 x = hx[rr][t];
        p[rr] = fmaf(x.x, w.x, p[rr]);
        p[rr] = fmaf(x.y, w.y, p[rr]);
        p[rr] = fmaf(x.z, w.z, p[rr]);
        p[rr] = fmaf(x.w, w.w, p[rr]);
      }
    }
    const bool b4 = lane & 16, b3 = lane & 8;
    const float a01 = (b4 ? p[1] : p[0]) + __shfl_xor_sync(0xffffffffu, b4 ? p[0] : p[1], 16);
    const float a23 = (b4 ? p[3] : p[2]) + __shfl_xor_sync(0xffffffffu, b4 ? p[2] : p[3], 16);
    float c = (b3 ? a23 : a01) + __shfl_xor_sync(0xffffffffu, b3 ? a01 : a23, 8);
    c += __shfl_xor_sync(0xffffffffu, c, 4);
    c += __shfl_xor_sync(0xffffffffu, c, 2);
    c += __shfl_xor_sync(0xffffffffu, c, 1);
    return c;
  };
  for (long r0 = ((long)blockIdx.x * wpb + warp) * 4; r0 < R; r0 += (long)gridDim.x * wpb * 4) {
    // the two streams one after the other (64 data registers instead of 128: two blocks per SM)
    float4 hx[4][T];
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const long r = r0 + rr < R ? r0 + rr : R - 1;
      const float4* h = reinterpret_cast<const float4*>(H + r * (2 * HID));
#pragma unroll
      for (int t = 0; t < T; ++t) hx[rr][t] = __ldg(h + lane + 32 * t);
    }
    const float v = dot4(hx, 0) + bz[0];
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const long r = r0 + rr < R ? r0 + rr : R - 1;
      const float4* h = reinterpret_cast<const float4*>(H + r * (2 * HID)) + HID / 4;
#pragma unroll
      for (int t = 0; t < T; ++t) hx[rr][t] = __ldg(h + lane + 32 * t);
    }
    float asum = 0.f, mine0 = 0.f, mine1 = 0.f, mine2 = 0.f;
    for (int k = 1; k <= A; ++k) {
      const float c = dot4(hx, k) + bz[k];
      asum += c;
      const int a = k - 1;
      if ((a & 7) == my_j) {                          // A <= 24 on this path
        if (a < 8) mine0 = c; else if (a < 16) mine1 = c; else mine2 = c;
      }
    }
    const long r = r0 + my_rr;
    if (r < R) {
      const long b = r / Nq, qi = r - b * Nq;                 // sample-major row -> quantile-major output row
      float* out = q + (qi * B + b) * A;
#pragma unroll
      for (int g = 0; g < 3; ++g) {
        const int a = my_j + 8 * g;
        const float mg = g == 0 ? mine0 : (g == 1 ? mine1 : mine2);
        if (a < A) out[a] = v + mg - asum / (float)A;
      }
    }
  }
}

// The same arithmetic (same operation order per output: bit-identical q) with the rows streamed through shared memory.
// Every warp owns one 4-row stage (4 x 2*HID floats, contiguous in H) filled by a bulk async copy that completes on the
// warp's mbarrier; as soon as the advantage halves of the current rows sit in registers, lane 0 launches the copy of the
// warp's next 4 rows, which then runs under the A advantage products (95 % of the arithmetic).  The row registers are no
// longer the only bytes in flight, so one CTA per SM (zs_warps: 8 warps at HID = 512) keeps HBM busy, and with the
// register cap gone the advantage loop runs two independent product / shuffle chains at a time.
__device__ __forceinline__ uint32_t zs_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void zs_bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(zs_smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   zs_smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(zs_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void zs_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "ZS_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra ZS_DONE_%=;\n"
      "bra ZS_WAIT_%=;\n"
      "ZS_DONE_%=:\n"
      "}\n" ::"r"(zs_smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// Warps per CTA: as many 4-row stages as fit in 128 KB (8 at HID = 512), at most 16.  The bytes in flight per SM stay at
// 128 KB for every width from 256 up, and the z-weights keep room beside them.
template <int HID>
constexpr int zs_warps() { return 4096 / HID < 16 ? 4096 / HID : 16; }
template <int HID>
constexpr size_t zs_smem_bytes(int A) {
  return (size_t)zs_warps<HID>() * 4 * 2 * HID * sizeof(float) + (size_t)(1 + A) * HID * sizeof(float) + 32 * sizeof(float) +
         zs_warps<HID>() * sizeof(uint64_t);
}

template <int HID>
__global__ void __launch_bounds__(zs_warps<HID>() * 32, 1) z_dueling_fwd4s_kernel(long R, int B, int A,
                                                                                 const float* __restrict__ H,
                                                                                 const float* __restrict__ Wz,
                                                                                 const float* __restrict__ bz, float* __restrict__ q) {
  constexpr int ZS_WARPS = zs_warps<HID>();
  extern __shared__ __align__(1024) unsigned char zs_raw[];
  constexpr int ROW = 2 * HID;                                  // floats per row of H
  float* stage_all = reinterpret_cast<float*>(zs_raw);          // ZS_WARPS x (4 rows)
  float* sW = stage_all + ZS_WARPS * 4 * ROW;                   // (1+A) * HID
  float* sB = sW + (1 + A) * HID;                               // 32
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + 32);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < (1 + A) * HID / 4; i += blockDim.x)
    reinterpret_cast<float4*>(sW)[i] = reinterpret_cast<const float4*>(Wz)[i];
  if (threadIdx.x < 32) sB[threadIdx.x] = threadIdx.x <= A ? bz[threadIdx.x] : 0.f;
  if (threadIdx.x < ZS_WARPS)
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(zs_smem_u32(bars + threadIdx.x)), "r"(1));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  constexpr int T = HID / 128;
  const int Nq = (int)(R / B);
  const int my_rr = ((lane >> 3) & 1) * 2 + ((lane >> 4) & 1), my_j = lane & 7;
  float* stage = stage_all + warp * 4 * ROW;
  uint64_t* bar = bars + warp;
  auto issue = [&](long r) {
    const long left = R - r;
    zs_bulk_load(stage, H + r * ROW, (uint32_t)((left < 4 ? left : 4) * ROW * sizeof(float)), bar);
  };
  // the transpose-reduce of z_dueling_fwd4_kernel: lane l ends with the sum of row rr(l)
  auto fold = [&](const float (&p)[4]) -> float {
    const bool b4 = lane & 16, b3 = lane & 8;
    const float a01 = (b4 ? p[1] : p[0]) + __shfl_xor_sync(0xffffffffu, b4 ? p[0] : p[1], 16);
    const float a23 = (b4 ? p[3] : p[2]) + __shfl_xor_sync(0xffffffffu, b4 ? p[2] : p[3], 16);
    float c = (b3 ? a23 : a01) + __shfl_xor_sync(0xffffffffu, b3 ? a01 : a23, 8);
    c += __shfl_xor_sync(0xffffffffu, c, 4);
    c += __shfl_xor_sync(0xffffffffu, c, 2);
    c += __shfl_xor_sync(0xffffffffu, c, 1);
    return c;
  };
  auto dot4 = [&](const float4 (&hx)[4][T], int k) -> float {
    const float4* wk = reinterpret_cast<const float4*>(sW + k * HID);
    float p[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const float4 w = wk[lane + 32 * t];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const float4 x = hx[rr][t];
        p[rr] = fmaf(x.x, w.x, p[rr]);
        p[rr] = fmaf(x.y, w.y, p[rr]);
        p[rr] = fmaf(x.z, w.z, p[rr]);
        p[rr] = fmaf(x.w, w.w, p[rr]);
      }
    }
    return fold(p);
  };
  const long stride = (long)gridDim.x * ZS_WARPS * 4;
  long r0 = ((long)blockIdx.x * ZS_WARPS + warp) * 4;
  if (r0 < R && lane == 0) issue(r0);
  uint32_t parity = 0;
  for (; r0 < R; r0 += stride) {
    zs_wait(bar, parity);
    parity ^= 1;
    float4 hx[4][T];
#pragma unroll
    for (int rr = 0; rr < 4; ++rr)
#pragma unroll
      for (int t = 0; t < T; ++t) hx[rr][t] = reinterpret_cast<const float4*>(stage + rr * ROW)[lane + 32 * t];
    const float v = dot4(hx, 0) + sB[0];
#pragma unroll
    for (int rr = 0; rr < 4; ++rr)
#pragma unroll
      for (int t = 0; t < T; ++t) hx[rr][t] = reinterpret_cast<const float4*>(stage + rr * ROW + HID)[lane + 32 * t];
    __syncwarp();                                       // every lane has its copy of the rows: the stage is free
    if (lane == 0 && r0 + stride < R) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      issue(r0 + stride);
    }
    float asum = 0.f, mine0 = 0.f, mine1 = 0.f, mine2 = 0.f;
    auto keep = [&](int a, float c) {                   // A <= 24 on this path
      if ((a & 7) == my_j) {
        if (a < 8) mine0 = c; else if (a < 16) mine1 = c; else mine2 = c;
      }
    };
    int k = 1;
    for (; k + 1 <= A; k += 2) {                        // two independent chains; asum still adds in order k, k+1
      const float c0 = dot4(hx, k) + sB[k];
      const float c1 = dot4(hx, k + 1) + sB[k + 1];
      asum += c0;
      asum += c1;
      keep(k - 1, c0);
      keep(k, c1);
    }
    if (k <= A) {
      const float c = dot4(hx, k) + sB[k];
      asum += c;
      keep(k - 1, c);
    }
    const long r = r0 + my_rr;
    if (r < R) {
      const long b = r / Nq, qi = r - b * Nq;                 // sample-major row -> quantile-major output row
      float* out = q + (qi * B + b) * A;
#pragma unroll
      for (int g = 0; g < 3; ++g) {
        const int a = my_j + 8 * g;
        const float mg = g == 0 ? mine0 : (g == 1 ? mine1 : mine2);
        if (a < A) out[a] = v + mg - asum / (float)A;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Double-DQN action: a*[b] = argmax_a mean_k q[k*B+b, a]               (compute_loss_iqn.py:238-245)
// ------------------------------------------------------------------------------------------------
__global__ void argmax_mean_kernel(int B, int K, int A, const float* __restrict__ q, int64_t* __restrict__ a_star) {
  // one warp per transition, lane a (< A <= 32) sums its action's K quantile values in order k = 0..K-1
  const int b = (int)(((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  float s = -INFINITY;
  if (lane < A) {
    s = 0.f;
    for (int k = 0; k < K; ++k) s += q[((long)k * B + b) * A + lane];
    s /= (float)K;
  }
  // argmax with the first maximal index winning (torch.argmax)
  float best = s;
  int arg = lane;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
  }
  if (lane == 0) a_star[b] = arg;
}

// ------------------------------------------------------------------------------------------------
// Fused IQN quantile-Huber loss, forward + dloss/dtheta            (compute_loss_iqn.py:262-357)
//   T[b,j]   = R[b] + fl(gamma^n)*nt[b] * q_tgt[(j*B+b), a*[b]]
//   th[b,i]  = q_on[(i*B+b), act[b]]
//   loss[b]  = (1/N') sum_j sum_i |tau_i - 1{d<0}| * huber_k(d) / k ,  d = T_j - th_i
//   dth[i*B+b] = dloss[b]/dth_i  (indicator detached, :344-346)
// One CTA per transition; thread i owns th_i and walks the N' targets staged in shared memory.
// ------------------------------------------------------------------------------------------------
__global__ void iqn_loss_kernel(int B, int N, int Np, int A, const float* __restrict__ q_on,
                                const float* __restrict__ q_tgt, const float* __restrict__ tau,
                                const int64_t* __restrict__ actions, const int64_t* __restrict__ a_star,
                                const float* __restrict__ returns, const float* __restrict__ nonterminals,
                                float gamma_n, float kappa, float* __restrict__ loss, float* __restrict__ dtheta,
                                float* __restrict__ theta_out, float* __restrict__ target_out) {
  extern __shared__ float sT[];  // Np targets + 32 reduction slots
  float* red = sT + Np;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int as = (int)a_star[b], ac = (int)actions[b];
  const float g = __fmul_rn(gamma_n, nonterminals[b]);
  for (int j = tid; j < Np; j += blockDim.x) {
    const float t = __fadd_rn(returns[b], __fmul_rn(g, q_tgt[((long)j * B + b) * A + as]));
    sT[j] = t;
    if (target_out) target_out[(long)b * Np + j] = t;
  }
  __syncthreads();
  float part = 0.f;
  for (int i = tid; i < N; i += blockDim.x) {
    const float th = q_on[((long)i * B + b) * A + ac];
    const float ta = tau[(long)i * B + b];
    float acc = 0.f, gacc = 0.f;
    for (int j = 0; j < Np; ++j) {
      const float d = sT[j] - th;
      const float ad = fabsf(d);
      const float hub = ad <= kappa ? 0.5f * d * d : kappa * (ad - 0.5f * kappa);
      const float dh = ad <= kappa ? d : copysignf(kappa, d);
      const float w = fabsf(ta - (d < 0.f ? 1.f : 0.f));
      acc += w * hub / kappa;
      gacc -= w * dh / kappa;
    }
    part += acc;
    dtheta[(long)i * B + b] = gacc / (float)Np;
    if (theta_out) theta_out[(long)b * N + i] = th;
  }
  part = warp_sum(part);
  if ((tid & 31) == 0) red[tid >> 5] = part;
  __syncthreads();
  if (tid < 32) {
    float v = tid < (blockDim.x >> 5) ? red[tid] : 0.f;
    v = warp_sum(v);
    if (tid == 0) loss[b] = v / (float)Np;
  }
}

// ------------------------------------------------------------------------------------------------
// Backward of dueling + z-layers + hidden ReLU, one warp per row.
//   g = dtheta[r] * gscale[b];  dq[a] = g*1{a==act}  =>  dv = g ,  da_k = g*(1{k==act} - 1/A)
//   dH_v = dv * w_zv ; dH_a = g*(W_za[act] - colmean(W_za)) ; masked by H > 0
//   dz (R, 32): [g, da_0..da_{A-1}, 0...] feeds the z-layer weight-gradient reduction.
// ------------------------------------------------------------------------------------------------
template <int HID>
__global__ void z_dueling_bwd_kernel(long R, int B, int A, const float* __restrict__ H, const float* __restrict__ Wz,
                                     const float* __restrict__ dtheta, const float* __restrict__ gscale, float gmul,
                                     const int64_t* __restrict__ actions, float* __restrict__ dH,
                                     float* __restrict__ dz, __nv_bfloat16* __restrict__ dz_bf) {
  extern __shared__ float sW[];  // (1+A)*HID weights + HID colmean
  float* wbar = sW + (1 + A) * HID;
  for (int i = threadIdx.x; i < (1 + A) * HID; i += blockDim.x) sW[i] = Wz[i];
  __syncthreads();
  for (int j = threadIdx.x; j < HID; j += blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < A; ++k) s += sW[(1 + k) * HID + j];
    wbar[j] = s / (float)A;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  for (long r = (long)blockIdx.x * wpb + warp; r < R; r += (long)gridDim.x * wpb) {
    const int Nq = (int)(R / B);
    const int b = (int)(r / Nq);                            // sample-major rows; dtheta arrives quantile-major
    const float g = dtheta[(r - (long)b * Nq) * B + b] * (gscale[b] * gmul);
    const int act = (int)actions[b];
    const float* h = H + r * (2 * HID);
    float* o = dH + r * (2 * HID);
    const float* wa = sW + (1 + act) * HID;
    for (int j = lane; j < HID; j += 32) {
      o[j] = h[j] > 0.f ? g * sW[j] : 0.f;
      o[HID + j] = h[HID + j] > 0.f ? g * (wa[j] - wbar[j]) : 0.f;
    }
    float z = 0.f;
    if (lane == 0) z = g;
    else if (lane <= A) z = g * ((lane - 1 == act ? 1.f : 0.f) - 1.f / (float)A);
    dz[r * 32 + lane] = z;
    if (dz_bf) dz_bf[r * 32 + lane] = __float2bfloat16_rn(z);
  }
}

// bf16-operand variant: the data gradient leaves directly as the two bf16 images the tensor-core products consume
// (dh_hi (R, 2*HID) for the dgrad, dh_hiT (2*HID, R) for the wgrad) plus its fp32 column sums (bias gradients); the fp32
// dH matrix is never written.  One block = 32 consecutive rows; a row is 2*HID/8 chunks of 8 columns, HC = HID/128 per
// lane.  The transposed image goes through an XOR-swizzled shared tile (16-byte chunk c/8 of row r sits in slot
// (c/8) ^ ((r >> 3) & 3)) and leaves as 64-byte column segments; the tile exists only when dh_hiT is requested.
template <int HID>
__global__ void __launch_bounds__(256) z_dueling_bwd_bf16_kernel(long R, int B, int A, const float* __restrict__ H,
                                                                 const __nv_bfloat16* __restrict__ Hb,
                                                                 const float* __restrict__ Wz,
                                                                 const float* __restrict__ dtheta,
                                                                 const float* __restrict__ gscale, float gmul,
                                                                 const int64_t* __restrict__ actions,
                                                                 __nv_bfloat16* __restrict__ dh_hi,
                                                                 __nv_bfloat16* __restrict__ dh_hiT,
                                                                 float* __restrict__ colsum, float* __restrict__ dz,
                                                                 __nv_bfloat16* __restrict__ dz_bf) {
  constexpr int HC = HID / 128;                        // 8-column chunks per lane and row
  constexpr int NCH = 2 * HID / 8;                     // chunks per row
  extern __shared__ __align__(16) float sW[];          // (1+A)*HID weights | HID colmean | 2*HID column sums | tile
  float* wbar = sW + (1 + A) * HID;
  float* cs = wbar + HID;
  uint4* tile = reinterpret_cast<uint4*>(cs + 2 * HID);   // [32 rows][NCH chunks of 8 bf16], only if dh_hiT != NULL
  for (int i = threadIdx.x; i < (1 + A) * HID / 4; i += blockDim.x)
    reinterpret_cast<float4*>(sW)[i] = reinterpret_cast<const float4*>(Wz)[i];
  for (int i = threadIdx.x; i < 2 * HID; i += blockDim.x) cs[i] = 0.f;
  __syncthreads();
  for (int j = threadIdx.x; j < HID; j += blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < A; ++k) s += sW[(1 + k) * HID + j];
    wbar[j] = s / (float)A;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Nq = (int)(R / B);
  float bs[HC][8];
#pragma unroll
  for (int it = 0; it < HC; ++it)
#pragma unroll
    for (int i = 0; i < 8; ++i) bs[it][i] = 0.f;
  const long n_blk = (R + 31) / 32;
  for (long blk = blockIdx.x; blk < n_blk; blk += gridDim.x) {   // persistent: column sums stay in registers
  const long r0 = blk * 32;
  for (int rr = 0; rr < 4; ++rr) {
    const int rl = warp * 4 + rr;
    const long r = r0 + rl;
    const bool ok = r < R;
    const long rc = ok ? r : 0;
    const int b = (int)(rc / Nq);                            // sample-major rows; dtheta arrives quantile-major
    const float g = ok ? dtheta[(rc - (long)b * Nq) * B + b] * (gscale[b] * gmul) : 0.f;
    const int act = (int)actions[b];
    const float* wa = sW + (1 + act) * HID;
    // the ReLU mask only needs the SIGN of h: read the bf16 image when the forward left one (half the bytes); all of
    // a row's loads are issued before the first use
    float hrow[HC][8];
#pragma unroll
    for (int it = 0; it < HC; ++it) {
      const int c0 = (lane + 32 * it) * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) hrow[it][i] = 0.f;
      if (ok) {
        if (Hb != nullptr) {
          const uint4 u = __ldg(reinterpret_cast<const uint4*>(Hb + r * (2 * HID) + c0));
          const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            hrow[it][2 * i] = __uint_as_float(w4[i] << 16);
            hrow[it][2 * i + 1] = __uint_as_float(w4[i] & 0xffff0000u);
          }
        } else {
          const float4 a = __ldg(reinterpret_cast<const float4*>(H + r * (2 * HID) + c0));
          const float4 c = __ldg(reinterpret_cast<const float4*>(H + r * (2 * HID) + c0 + 4));
          hrow[it][0] = a.x; hrow[it][1] = a.y; hrow[it][2] = a.z; hrow[it][3] = a.w;
          hrow[it][4] = c.x; hrow[it][5] = c.y; hrow[it][6] = c.z; hrow[it][7] = c.w;
        }
      }
    }
#pragma unroll
    for (int it = 0; it < HC; ++it) {
      const int chunk = lane + 32 * it, c0 = chunk * 8;
      const float (&hv)[8] = hrow[it];
      float val[8];
      // chunk group it covers columns [256*it, 256*it + 256): wholly one stream unless HID / 256 is not whole (384, 640,
      // 896), where one group straddles the two streams and each lane picks its own
      const bool value = (it + 1) * 256 <= HID ? true : (it * 256 >= HID ? false : c0 < HID);
      if (value) {                                             // value stream: dv * w_zv
#pragma unroll
        for (int i = 0; i < 8; ++i) val[i] = hv[i] > 0.f ? g * sW[c0 + i] : 0.f;
      } else {                                                 // advantage stream: g * (W_za[act] - colmean)
        const int j0 = c0 - HID;
#pragma unroll
        for (int i = 0; i < 8; ++i) val[i] = hv[i] > 0.f ? g * (wa[j0 + i] - wbar[j0 + i]) : 0.f;
      }
      uint32_t w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h2 = __floats2bfloat162_rn(val[2 * i], val[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t*>(&h2);
        bs[it][2 * i] += val[2 * i];
        bs[it][2 * i + 1] += val[2 * i + 1];
      }
      const uint4 pk = make_uint4(w[0], w[1], w[2], w[3]);
      if (ok) *reinterpret_cast<uint4*>(dh_hi + r * (2 * HID) + c0) = pk;
      if (dh_hiT) tile[rl * NCH + (chunk ^ ((rl >> 3) & 3))] = pk;
    }
    if (ok) {
      float z = 0.f;
      if (lane == 0) z = g;
      else if (lane <= A) z = g * ((lane - 1 == act ? 1.f : 0.f) - 1.f / (float)A);
      dz[r * 32 + lane] = z;
      if (dz_bf) dz_bf[r * 32 + lane] = __float2bfloat16_rn(z);     // (R, 32) row-major: MN-major operand of dWz
    }
  }
  if (dh_hiT == nullptr) continue;                               // (warp-uniform) no transposed image wanted
  __syncthreads();
  // transposed image: item = (column c, piece p of 8 rows); a warp covers 8 columns x 4 pieces = 8 x 64 contiguous bytes
  const unsigned short* t16 = reinterpret_cast<const unsigned short*>(tile);
  for (int item = threadIdx.x; item < 2 * HID * 4; item += blockDim.x) {
    const int c = item >> 2, piece = item & 3;
    if (r0 + 8 * piece + 7 < R) {
      const int slot = (c >> 3) ^ piece;
      uint32_t w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const unsigned short lo = t16[((8 * piece + 2 * i) * NCH + slot) * 8 + (c & 7)];
        const unsigned short hi = t16[((8 * piece + 2 * i + 1) * NCH + slot) * 8 + (c & 7)];
        w[i] = (uint32_t)lo | ((uint32_t)hi << 16);
      }
      *reinterpret_cast<uint4*>(dh_hiT + (long)c * R + r0 + 8 * piece) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
  __syncthreads();                                               // the tile is rewritten by the next row block
  }
#pragma unroll
  for (int it = 0; it < HC; ++it)
#pragma unroll
    for (int i = 0; i < 8; ++i) atomicAdd(&cs[(lane + 32 * it) * 8 + i], bs[it][i]);
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * HID; c += blockDim.x) atomicAdd(&colsum[c], cs[c]);
}

// dWz (32, 2*HID) from dz^T * H  ->  parameter gradients of the two noisy z-layers.
//   z_v: weight (1,HID) = dWz[0, :HID] ; z_a: weight (A,HID) = dWz[1+k, HID:]
//   dmu += g ; dsigma += g * eps          (model.py:45-53)
__global__ void z_wgrad_finish_kernel(int A, int HID, const float* __restrict__ dWz, const float* __restrict__ dbz,
                                      const float* __restrict__ eps_w_zv, const float* __restrict__ eps_b_zv,
                                      const float* __restrict__ eps_w_za, const float* __restrict__ eps_b_za,
                                      float* g_mu_zv, float* g_sig_zv, float* g_bmu_zv, float* g_bsig_zv,
                                      float* g_mu_za, float* g_sig_za, float* g_bmu_za, float* g_bsig_za) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < HID) {
    const float g = dWz[idx];
    g_mu_zv[idx] += g;
    g_sig_zv[idx] += g * eps_w_zv[idx];
  }
  if (idx < A * HID) {
    const int k = idx / HID, j = idx % HID;
    const float g = dWz[(long)(1 + k) * (2 * HID) + HID + j];
    g_mu_za[idx] += g;
    g_sig_za[idx] += g * eps_w_za[idx];
  }
  if (idx == 0) {
    g_bmu_zv[0] += dbz[0];
    g_bsig_zv[0] += dbz[0] * eps_b_zv[0];
  }
  if (idx < A) {
    g_bmu_za[idx] += dbz[1 + idx];
    g_bsig_za[idx] += dbz[1 + idx] * eps_b_za[idx];
  }
}

// dmu_b += db ; dsigma_b += db * eps_b
__global__ void noisy_bias_grad_kernel(int n, const float* __restrict__ db, const float* __restrict__ eps_b,
                                       float* g_bmu, float* g_bsig) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  g_bmu[i] += db[i];
  g_bsig[i] += db[i] * eps_b[i];
}

// ------------------------------------------------------------------------------------------------
// Backward through x = feat[b] (.) phi[r]  (model.py:149-151) given dX (in place -> dpre):
//   dpre[r,f]  = dX * feat[b,f] * 1{phi>0}          (grad wrt iqn_fc pre-activation)
//   dfeat[b,f] = sum_q dX[q*B+b,f] * phi[q*B+b,f]   with phi = X/feat where feat > 0
// (feat == 0 means conv3's ReLU is closed, so dfeat there is masked anyway.)
// ------------------------------------------------------------------------------------------------
__global__ void embed_bwd_elem_kernel(int B, int Nq, int F, const float* __restrict__ X, const float* __restrict__ feat,
                                      float* __restrict__ dX, float* __restrict__ dfeat) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)B * F) return;
  const float ft = feat[idx];
  float acc = 0.f;
  for (int q = 0; q < Nq; ++q) {
    const long bb = idx / F;
    const long o = ((bb * Nq + q) * F) + (idx - bb * F);     // sample-major rows
    const float x = X[o], dx = dX[o];
    acc = fmaf(dx, x, acc);
    dX[o] = x > 0.f ? dx * ft : 0.f;
  }
  dfeat[idx] = ft > 0.f ? acc / ft : 0.f;
}

// ------------------------------------------------------------------------------------------------
// Adam over a flat fp32 arena (torch.optim.Adam semantics; agent.py:43, learner.py:24)
// ------------------------------------------------------------------------------------------------
__global__ void adam_kernel(long n, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, float neg_step_size, float sqrt_bc2, float eps, float b1, float b2,
                            float grad_scale, const riqn_dyn_state* __restrict__ dyn) {
  if (dyn) { neg_step_size = dyn->adam_neg_step_size; sqrt_bc2 = dyn->adam_sqrt_bc2; }
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float gi = g[i] * grad_scale;
    const float mi = m[i] + (gi - m[i]) * (1.f - b1);           // lerp_, as torch
    const float vi = v[i] * b2 + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), sqrt_bc2), eps);   // (v.sqrt() / sqrt(bc2)).add_(eps)
    p[i] = __fadd_rn(p[i], __fdiv_rn(__fmul_rn(neg_step_size, mi), denom)); // addcdiv_(m, denom, value=-step_size)
  }
}

static inline int grid_for(long total, int per = 256) {
  long b = (total + per - 1) / per;
  return (int)(b > 148L * 64 ? 148L * 64 : (b < 1 ? 1 : b));
}

}  // namespace riqn

using namespace riqn;

RIQN_API int riqn_fill_uniform(long n, unsigned long long seed, unsigned long long stream_id, float* out,
                               const riqn_dyn_state* dyn, void* stream) {
  riqn::note_launches(1);
  if (n <= 0) return 0;
  fill_uniform_kernel<<<riqn_cdiv((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(n, seed, stream_id, out, dyn);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_noisy_sample(long n, unsigned long long seed, unsigned long long stream_id, float* out,
                               const riqn_dyn_state* dyn, void* stream) {
  riqn::note_launches(1);
  if (n <= 0) return 0;
  fill_scaled_normal_kernel<<<riqn_cdiv((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(n, seed, stream_id, out, dyn);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_noisy_compose(int out_features, int in_features, const float* weight_mu, const float* weight_sigma,
                                float* weight_epsilon, const float* eps_in, const float* eps_out, const float* bias_mu,
                                const float* bias_sigma, float* bias_epsilon, float* w_eff, float* b_eff, int training,
                                void* stream) {
  riqn::note_launches(1);
  noisy_compose_kernel<<<grid_for((long)out_features * in_features), 256, 0, (cudaStream_t)stream>>>(
      out_features, in_features, weight_mu, weight_sigma, weight_epsilon, eps_in, eps_out, bias_mu, bias_sigma,
      bias_epsilon, w_eff, b_eff, training);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_noisy_reset_net(int n_layers, const riqn_noisy_layer* layers, unsigned long long seed, int sample,
                                  int training, const riqn_dyn_state* dyn, void* stream) {
  if (n_layers < 1 || n_layers > 8 || layers == nullptr) return (int)cudaErrorInvalidValue;
  cudaStream_t s = (cudaStream_t)stream;
  NoisyNet net;
  net.n = n_layers;
  for (int i = 0; i < n_layers; ++i) {
    net.l[i] = layers[i];
    const riqn_noisy_layer& L = layers[i];
    if (L.in_features % 4 || L.out_features < 1 || (reinterpret_cast<uintptr_t>(L.eps_in) & 15) ||
        (reinterpret_cast<uintptr_t>(L.weight_mu) & 15) || (reinterpret_cast<uintptr_t>(L.weight_sigma) & 15) ||
        (reinterpret_cast<uintptr_t>(L.weight_epsilon) & 15) || (reinterpret_cast<uintptr_t>(L.w_eff) & 15))
      return (int)cudaErrorInvalidValue;
  }
  if (sample) {
    riqn::note_launches(1);
    int blocks = 0;
    for (int i = 0; i < n_layers; ++i) {
      blocks += (int)riqn_cdiv((layers[i].in_features + 3) / 4, 256);
      net.blk_end[2 * i] = blocks;
      blocks += (int)riqn_cdiv((layers[i].out_features + 3) / 4, 256);
      net.blk_end[2 * i + 1] = blocks;
    }
    noisy_fill_net_kernel<<<blocks, 256, 0, s>>>(net, seed, dyn);
    RIQN_LAUNCH_CHECK();
  }
  riqn::note_launches(1);
  int blocks = 0;
  for (int i = 0; i < n_layers; ++i) {
    blocks += (int)riqn_cdiv((long)layers[i].out_features * (layers[i].in_features / 4), 256);
    net.blk_end[i] = blocks;
  }
  noisy_compose_net_kernel<<<blocks, 256, 0, s>>>(net, training);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_quantile_embed_fwd(int batch, int num_quantiles, int embed_dim, int feat_dim, const float* tau,
                                     const float* feat, const float* iqn_w, const float* iqn_b, float* cosv, float* x,
                                     void* stream) {
  riqn::note_launches(2);
  cudaStream_t s = (cudaStream_t)stream;
  const long R = (long)batch * num_quantiles;
  cos_embed_kernel<<<riqn_cdiv(R * embed_dim, 256), 256, 0, s>>>(batch, num_quantiles, embed_dim, tau, cosv);
  RIQN_LAUNCH_CHECK();
  EpiArgs e;
  e.bias = iqn_b;
  e.feat = feat;
  e.batch = num_quantiles;     // rows per sample (sample-major rows): feat row = m / num_quantiles
  return gemm_f32((int)R, feat_dim, embed_dim, cosv, embed_dim, 1, iqn_w, embed_dim, 1, x, feat_dim, EPI_EMBED, e, 1, s);
}

// Tensor-core embedding: cos -> bf16 (hi, lo); x = feat (.) relu(cos W_e^T + b_e) computed by the tcgen05 GEMM whose
// epilogue writes the bf16 operand images of x directly (x_hi/x_lo row-major for the head product, x_hiT/x_loT
// transposed for its weight gradient) and, only if x32 != NULL, the fp32 matrix.
RIQN_API int riqn_quantile_embed_fwd_tc(int batch, int num_quantiles, int embed_dim, int feat_dim, const float* tau,
                                        const float* feat, const void* iqn_w_hi, const void* iqn_w_lo, const float* iqn_b,
                                        void* cos_hi, void* cos_lo, void* cosT_hi, float* x32, void* x_hi, void* x_lo,
                                        void* x_hiT, void* x_loT, int x_fp16, void* stream) {
  riqn::note_launches(2);
  cudaStream_t s = (cudaStream_t)stream;
  const long R = (long)batch * num_quantiles;
  cos_embed_bf16_kernel<<<riqn_cdiv(R * embed_dim, 256), 256, 0, s>>>(batch, num_quantiles, embed_dim, tau, (__nv_bfloat16*)cos_hi,
                                                                     (__nv_bfloat16*)cos_lo, (__nv_bfloat16*)cosT_hi);
  RIQN_LAUNCH_CHECK();
  TcExtra ex;
  ex.feat = feat;
  ex.batch = num_quantiles;    // rows per sample
  ex.o_hi = (__nv_bfloat16*)x_hi;
  ex.o_lo = (__nv_bfloat16*)x_lo;
  ex.fmt = x_fp16 ? 4 : 0;       // x_hi = fp16(x) (head forward operand), x_lo (optional) = bf16(x) (backward operand)
  const bool want_t = x_hiT != nullptr || x_loT != nullptr;    // transposed images (cross-check arithmetic modes only)
  if (want_t && (x32 == nullptr || x_fp16)) return (int)cudaErrorInvalidValue;
  int rc = gemm_bf16_tc((int)R, feat_dim, embed_dim, (const __nv_bfloat16*)cos_hi, (const __nv_bfloat16*)cos_lo,
                        (const __nv_bfloat16*)iqn_w_hi, cos_lo ? (const __nv_bfloat16*)iqn_w_lo : nullptr, x32, feat_dim,
                        TC_EMBED, iqn_b, nullptr, nullptr, 1, s, &ex);
  if (rc == 0 && want_t) {
    riqn::note_launches(1);
    rc = split_bf16(R, feat_dim, x32, nullptr, nullptr, (__nv_bfloat16*)x_hiT, (__nv_bfloat16*)x_loT, s);
  }
  return rc;
}

// Backward on bf16 operands: dx (fp32, from the head dgrad) -> dfeat (overwritten), grad_iqn_b / grad_iqn_w accumulated.
// cos_hi (rows, embed_dim) bf16 row-major (the forward's image); dpre (rows, feat_dim) bf16 is workspace.  rows % 8 == 0.
RIQN_API int riqn_quantile_embed_bwd_tc(int batch, int num_quantiles, int embed_dim, int feat_dim, const void* x_hi,
                                        const void* x_lo, const float* feat, const void* cos_hi, const void* dx,
                                        int dx_is_bf16, void* dpre, float* dfeat, float* grad_iqn_w, float* grad_iqn_b,
                                        void* stream) {
  riqn::note_launches(2);
  cudaStream_t s = (cudaStream_t)stream;
  const long R = (long)batch * num_quantiles;
  if (R % 8 || feat_dim % 8 || embed_dim % 8) return (int)cudaErrorInvalidValue;
  if (num_quantiles % 2 == 0 && feat_dim % 4 == 0) {
    dim3 grid((feat_dim + 127) / 128, batch);
#define RIQN_EMB_BWD(DXB, XLO)                                                                                          \
  embed_bwd_wide_kernel<DXB, XLO><<<grid, 256, 0, s>>>(batch, num_quantiles, feat_dim, (const __nv_bfloat16*)x_hi,        \
                                                       (const __nv_bfloat16*)x_lo, feat, (const float*)dx,                \
                                                       (const __nv_bfloat16*)dx, (__nv_bfloat16*)dpre, dfeat, grad_iqn_b)
    if (dx_is_bf16 && feat_dim % 8 == 0) {
      dim3 grid8((feat_dim + 255) / 256, batch);
      if (x_lo)
        embed_bwd_wide8_kernel<true><<<grid8, 256, 0, s>>>(batch, num_quantiles, feat_dim, (const __nv_bfloat16*)x_hi,
                                                           (const __nv_bfloat16*)x_lo, feat, (const __nv_bfloat16*)dx,
                                                           (__nv_bfloat16*)dpre, dfeat, grad_iqn_b);
      else
        embed_bwd_wide8_kernel<false><<<grid8, 256, 0, s>>>(batch, num_quantiles, feat_dim, (const __nv_bfloat16*)x_hi,
                                                            nullptr, feat, (const __nv_bfloat16*)dx, (__nv_bfloat16*)dpre,
                                                            dfeat, grad_iqn_b);
    } else if (dx_is_bf16) { if (x_lo) RIQN_EMB_BWD(true, true); else RIQN_EMB_BWD(true, false); }
    else            { if (x_lo) RIQN_EMB_BWD(false, true); else RIQN_EMB_BWD(false, false); }
#undef RIQN_EMB_BWD
  } else {
    dim3 grid((feat_dim + 31) / 32, batch);
    embed_bwd_tile_kernel<<<grid, 256, 0, s>>>(batch, num_quantiles, feat_dim, (const __nv_bfloat16*)x_hi,
                                               (const __nv_bfloat16*)x_lo, feat, dx_is_bf16 ? nullptr : (const float*)dx,
                                               dx_is_bf16 ? (const __nv_bfloat16*)dx : nullptr, (__nv_bfloat16*)dpre, dfeat,
                                               grad_iqn_b);
  }
  RIQN_LAUNCH_CHECK();
  const int m_tiles = (feat_dim + 127) / 128;
  const int split = tc_pick_split(m_tiles, (R + 63) / 64);
  // dWe[f, i] += sum_r dpre[r, f] * cos[r, i]: both operands row-major, reduction over the rows (MN-major operands)
  TcExtra ex;
  ex.mn_major = 3;
  return gemm_bf16_tc(feat_dim, embed_dim, (int)R, (const __nv_bfloat16*)dpre, nullptr, (const __nv_bfloat16*)cos_hi, nullptr,
                      grad_iqn_w, embed_dim, TC_ATOMIC, nullptr, nullptr, nullptr, split, s, &ex);
}

RIQN_API int riqn_quantile_embed_bwd(int batch, int num_quantiles, int embed_dim, int feat_dim, const float* x,
                                     const float* feat, const float* cosv, float* dx_inout, float* dfeat,
                                     float* grad_iqn_w, float* grad_iqn_b, void* stream) {
  riqn::note_launches(3);
  cudaStream_t s = (cudaStream_t)stream;
  const long R = (long)batch * num_quantiles;
  embed_bwd_elem_kernel<<<riqn_cdiv((long)batch * feat_dim, 256), 256, 0, s>>>(batch, num_quantiles, feat_dim, x, feat,
                                                                             dx_inout, dfeat);
  RIQN_LAUNCH_CHECK();
  int rc = colsum_atomic(R, feat_dim, dx_inout, grad_iqn_b, s);
  if (rc) return rc;
  EpiArgs e;
  const int tiles = (feat_dim + 127) / 128;
  int split = (3 * 148 + tiles - 1) / tiles;
  if ((long)split * 64 > R) split = (int)((R + 63) / 64);
  // dWe[f, i] += sum_r dpre[r, f] * cos[r, i]
  return gemm_f32(feat_dim, embed_dim, (int)R, dx_inout, 1, feat_dim, cosv, 1, embed_dim, grad_iqn_w, embed_dim,
                  EPI_ATOMIC, e, split, s);
}

RIQN_API int riqn_noisy_linear_fwd(long rows, int in_features, int out_features, const float* x, const float* w_eff,
                                   const float* b_eff, float* h, void* stream) {
  riqn::note_launches(1);
  EpiArgs e;
  e.bias = b_eff;
  return gemm_f32((int)rows, out_features, in_features, x, in_features, 1, w_eff, in_features, 1, h, out_features,
                  EPI_BIAS_RELU, e, 1, (cudaStream_t)stream);
}

RIQN_API int riqn_noisy_linear_dgrad(long rows, int in_features, int out_features, const float* dh, const float* w_eff,
                                     float* dx, void* stream) {
  riqn::note_launches(1);
  EpiArgs e;
  return gemm_f32((int)rows, in_features, out_features, dh, out_features, 1, w_eff, 1, in_features, dx, in_features,
                  EPI_STORE, e, 1, (cudaStream_t)stream);
}

RIQN_API int riqn_noisy_linear_wgrad(long rows, int in_features, int out_features, const float* dh, const float* x,
                                     const float* weight_epsilon, const float* bias_epsilon, float* db_scratch,
                                     float* grad_weight_mu, float* grad_weight_sigma, float* grad_bias_mu,
                                     float* grad_bias_sigma, void* stream) {
  riqn::note_launches(3);
  cudaStream_t s = (cudaStream_t)stream;
  EpiArgs e;
  e.out2 = grad_weight_sigma;
  e.eps = weight_epsilon;
  int rc = gemm_f32(out_features, in_features, (int)rows, dh, 1, out_features, x, 1, in_features, grad_weight_mu,
                    in_features, EPI_NOISY_WGRAD, e, 1, s);
  if (rc) return rc;
  RIQN_CUDA(cudaMemsetAsync(db_scratch, 0, sizeof(float) * out_features, s));
  rc = colsum_atomic(rows, out_features, dh, db_scratch, s);
  if (rc) return rc;
  noisy_bias_grad_kernel<<<riqn_cdiv(out_features, 256), 256, 0, s>>>(out_features, db_scratch, bias_epsilon,
                                                                    grad_bias_mu, grad_bias_sigma);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_noisy_bias_grad(long rows, int out_features, const float* dh, const float* bias_epsilon,
                                  float* db_scratch, float* grad_bias_mu, float* grad_bias_sigma, void* stream) {
  riqn::note_launches(dh ? 2 : 1);
  cudaStream_t s = (cudaStream_t)stream;
  if (dh) {            // dh == NULL: db_scratch already holds the column sums (riqn_dueling_bwd_bf16)
    RIQN_CUDA(cudaMemsetAsync(db_scratch, 0, sizeof(float) * out_features, s));
    int rc = colsum_atomic(rows, out_features, dh, db_scratch, s);
    if (rc) return rc;
  }
  noisy_bias_grad_kernel<<<riqn_cdiv(out_features, 256), 256, 0, s>>>(out_features, db_scratch, bias_epsilon,
                                                                    grad_bias_mu, grad_bias_sigma);
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// z-layer + dueling entry points: one instantiation per supported width (every multiple of 128 up to 1024), each with
// its own per-device attribute cache.  A (width, A) pair whose shared memory does not fit is refused before any launch.
// ------------------------------------------------------------------------------------------------
namespace riqn {
constexpr size_t kMaxSmemOptin = 227 * 1024;   // opt-in dynamic shared memory per block on sm_100a

static inline bool hidden_supported(int hidden) { return hidden >= 128 && hidden <= 1024 && hidden % 128 == 0; }

static inline size_t dueling_bwd_bf16_smem(int hidden, int A, bool transposed) {
  return sizeof(float) * ((size_t)(1 + A) * hidden + hidden + 2 * hidden) + (transposed ? (size_t)32 * (2 * hidden / 8) * 16 : 0);
}

template <int HID>
static int dueling_fwd_launch(long rows, int batch, int A, const float* h, const float* wz, const float* bz, float* q,
                              cudaStream_t s) {
  const size_t smem = sizeof(float) * (1 + A) * HID;
  const int dev = PerDeviceOnce::device();
  if (A <= 24) {
    if (rows >= 4096 && (reinterpret_cast<uintptr_t>(h) & 15) == 0 && zs_smem_bytes<HID>(A) <= kMaxSmemOptin) {
      static PerDeviceOnce attrs_once;                                       // streamed variant: one CTA per SM
      if (!attrs_once.done[dev]) {
        const size_t most = zs_smem_bytes<HID>(24) < kMaxSmemOptin ? zs_smem_bytes<HID>(24) : kMaxSmemOptin;
        RIQN_CUDA(cudaFuncSetAttribute(z_dueling_fwd4s_kernel<HID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
        attrs_once.done[dev] = true;
      }
      z_dueling_fwd4s_kernel<HID><<<148, zs_warps<HID>() * 32, zs_smem_bytes<HID>(A), s>>>(rows, batch, A, h, wz, bz, q);
      return (int)cudaGetLastError();
    }
    static PerDeviceOnce attr4_once;
    if (!attr4_once.done[dev]) {
      RIQN_CUDA(cudaFuncSetAttribute(z_dueling_fwd4_kernel<HID>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(sizeof(float) * 25 * HID)));
      attr4_once.done[dev] = true;
    }
    z_dueling_fwd4_kernel<HID><<<148 * 2, 256, smem, s>>>(rows, batch, A, h, wz, bz, q);
  } else {
    static PerDeviceOnce attr_once;
    if (!attr_once.done[dev]) {
      RIQN_CUDA(cudaFuncSetAttribute(z_dueling_fwd_kernel<HID>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(sizeof(float) * 32 * HID)));
      attr_once.done[dev] = true;
    }
    z_dueling_fwd_kernel<HID><<<148 * 4, 256, smem, s>>>(rows, batch, A, h, wz, bz, q);
  }
  return (int)cudaGetLastError();
}

template <int HID>
static int dueling_bwd_launch(long rows, int batch, int A, const float* h, const float* wz, const float* dtheta,
                              const float* gscale, float gscale_mul, const long long* actions, float* dh, float* dz,
                              void* dz_bf16, cudaStream_t s) {
  const size_t smem = sizeof(float) * ((1 + A) * HID + HID);
  static PerDeviceOnce attr_once;
  const int dev = PerDeviceOnce::device();
  if (!attr_once.done[dev]) {
    RIQN_CUDA(cudaFuncSetAttribute(z_dueling_bwd_kernel<HID>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)(sizeof(float) * 33 * HID)));
    attr_once.done[dev] = true;
  }
  z_dueling_bwd_kernel<HID><<<148 * 4, 256, smem, s>>>(rows, batch, A, h, wz, dtheta, gscale, gscale_mul,
                                                        (const int64_t*)actions, dh, dz, (__nv_bfloat16*)dz_bf16);
  return (int)cudaGetLastError();
}

template <int HID>
static int dueling_bwd_bf16_launch(long rows, int batch, int A, const float* h, const void* h_bf16, const float* wz,
                                   const float* dtheta, const float* gscale, float gscale_mul, const long long* actions,
                                   void* dh_hi, void* dh_hi_t, float* dh_colsum, float* dz, void* dz_bf16, cudaStream_t s) {
  const size_t smem = dueling_bwd_bf16_smem(HID, A, dh_hi_t != nullptr);
  static PerDeviceOnce attr_once;
  const int dev = PerDeviceOnce::device();
  if (!attr_once.done[dev]) {
    const size_t most = dueling_bwd_bf16_smem(HID, 31, true) < kMaxSmemOptin ? dueling_bwd_bf16_smem(HID, 31, true) : kMaxSmemOptin;
    RIQN_CUDA(cudaFuncSetAttribute(z_dueling_bwd_bf16_kernel<HID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
    attr_once.done[dev] = true;
  }
  RIQN_CUDA(cudaMemsetAsync(dh_colsum, 0, sizeof(float) * 2 * HID, s));
  const long n_blk = (rows + 31) / 32;
  z_dueling_bwd_bf16_kernel<HID><<<(unsigned)(n_blk < 148 * 2 ? n_blk : 148 * 2), 256, smem, s>>>(
      rows, batch, A, h, (const __nv_bfloat16*)h_bf16, wz, dtheta, gscale, gscale_mul, (const int64_t*)actions,
      (__nv_bfloat16*)dh_hi, (__nv_bfloat16*)dh_hi_t, dh_colsum, dz, (__nv_bfloat16*)dz_bf16);
  return (int)cudaGetLastError();
}
}  // namespace riqn

#define RIQN_HIDDEN_DISPATCH(hidden, launch, ...)                                                                       \
  switch (hidden) {                                                                                                    \
    case 128: return launch<128>(__VA_ARGS__);                                                                         \
    case 256: return launch<256>(__VA_ARGS__);                                                                         \
    case 384: return launch<384>(__VA_ARGS__);                                                                         \
    case 512: return launch<512>(__VA_ARGS__);                                                                         \
    case 640: return launch<640>(__VA_ARGS__);                                                                         \
    case 768: return launch<768>(__VA_ARGS__);                                                                         \
    case 896: return launch<896>(__VA_ARGS__);                                                                         \
    case 1024: return launch<1024>(__VA_ARGS__);                                                                       \
    default: return (int)cudaErrorInvalidValue;                                                                        \
  }

RIQN_API int riqn_dueling_fwd(long rows, int batch, int hidden, int action_space, const float* h, const float* wz,
                              const float* bz, float* q, void* stream) {
  riqn::note_launches(1);
  if (!hidden_supported(hidden) || action_space < 1 || action_space > 31 ||
      sizeof(float) * (1 + action_space) * hidden > kMaxSmemOptin)
    return (int)cudaErrorInvalidValue;
  RIQN_HIDDEN_DISPATCH(hidden, dueling_fwd_launch, rows, batch, action_space, h, wz, bz, q, (cudaStream_t)stream);
}

RIQN_API int riqn_dueling_bwd(long rows, int batch, int hidden, int action_space, const float* h, const float* wz,
                              const float* dtheta, const float* gscale, float gscale_mul, const long long* actions, float* dh, float* dz,
                              void* dz_bf16, void* stream) {
  riqn::note_launches(1);
  if (!hidden_supported(hidden) || action_space < 1 || action_space > 31 ||
      sizeof(float) * ((1 + action_space) * hidden + hidden) > kMaxSmemOptin)
    return (int)cudaErrorInvalidValue;
  RIQN_HIDDEN_DISPATCH(hidden, dueling_bwd_launch, rows, batch, action_space, h, wz, dtheta, gscale, gscale_mul, actions, dh,
                       dz, dz_bf16, (cudaStream_t)stream);
}

RIQN_API int riqn_dueling_bwd_bf16(long rows, int batch, int hidden, int action_space, const float* h, const void* h_bf16,
                                   const float* wz,
                                   const float* dtheta, const float* gscale, float gscale_mul, const long long* actions, void* dh_hi,
                                   void* dh_hi_t, float* dh_colsum, float* dz, void* dz_bf16, void* stream) {
  riqn::note_launches(1);
  // the transposed image needs a (32 rows x 2*hidden) bf16 tile beside the weights: refused where it does not fit
  if (!hidden_supported(hidden) || action_space < 1 || action_space > 31 || rows % 8 ||
      dueling_bwd_bf16_smem(hidden, action_space, dh_hi_t != nullptr) > kMaxSmemOptin)
    return (int)cudaErrorInvalidValue;
  RIQN_HIDDEN_DISPATCH(hidden, dueling_bwd_bf16_launch, rows, batch, action_space, h, h_bf16, wz, dtheta, gscale, gscale_mul,
                       actions, dh_hi, dh_hi_t, dh_colsum, dz, dz_bf16, (cudaStream_t)stream);
}
#undef RIQN_HIDDEN_DISPATCH

RIQN_API int riqn_z_wgrad(long rows, int hidden, int action_space, const float* dz, const float* h, float* dwz_scratch,
                          float* dbz_scratch, const float* eps_w_zv, const float* eps_b_zv, const float* eps_w_za,
                          const float* eps_b_za, float* g_mu_zv, float* g_sig_zv, float* g_bmu_zv, float* g_bsig_zv,
                          float* g_mu_za, float* g_sig_za, float* g_bmu_za, float* g_bsig_za, void* stream) {
  riqn::note_launches(3);
  cudaStream_t s = (cudaStream_t)stream;
  const int W = 2 * hidden;
  RIQN_CUDA(cudaMemsetAsync(dwz_scratch, 0, sizeof(float) * 32 * W, s));
  RIQN_CUDA(cudaMemsetAsync(dbz_scratch, 0, sizeof(float) * 32, s));
  EpiArgs e;
  int split = 32;
  if ((long)split * 64 > rows) split = (int)((rows + 63) / 64);
  int rc = gemm_f32(32, W, (int)rows, dz, 1, 32, h, 1, W, dwz_scratch, W, EPI_ATOMIC, e, split, s);
  if (rc) return rc;
  rc = colsum_atomic(rows, 32, dz, dbz_scratch, s);
  if (rc) return rc;
  z_wgrad_finish_kernel<<<riqn_cdiv((long)action_space * hidden, 256), 256, 0, s>>>(
      action_space, hidden, dwz_scratch, dbz_scratch, eps_w_zv, eps_b_zv, eps_w_za, eps_b_za, g_mu_zv, g_sig_zv, g_bmu_zv,
      g_bsig_zv, g_mu_za, g_sig_za, g_bmu_za, g_bsig_za);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_z_wgrad_tc(long rows, int hidden, int action_space, const void* dz_bf16, const void* h_bf16, const float* dz,
                             float* dwz_scratch, float* dbz_scratch, const float* eps_w_zv, const float* eps_b_zv,
                             const float* eps_w_za, const float* eps_b_za, float* g_mu_zv, float* g_sig_zv, float* g_bmu_zv,
                             float* g_bsig_zv, float* g_mu_za, float* g_sig_za, float* g_bmu_za, float* g_bsig_za,
                             void* stream) {
  riqn::note_launches(3);
  cudaStream_t s = (cudaStream_t)stream;
  const int W = 2 * hidden;
  if (rows % 8) return (int)cudaErrorInvalidValue;
  RIQN_CUDA(cudaMemsetAsync(dwz_scratch, 0, sizeof(float) * 32 * W, s));
  RIQN_CUDA(cudaMemsetAsync(dbz_scratch, 0, sizeof(float) * 32, s));
  const int n_tiles = (W + 255) / 256;
  const int split = tc_pick_split(n_tiles, (rows + 63) / 64);
  // dWz[z, j] = sum_r dz[r, z] * h[r, j]: both operands row-major, reduction over the rows (MN-major operands)
  TcExtra ex;
  ex.mn_major = 3;
  int rc = gemm_bf16_tc(32, W, (int)rows, (const __nv_bfloat16*)dz_bf16, nullptr, (const __nv_bfloat16*)h_bf16, nullptr,
                        dwz_scratch, W, TC_ATOMIC, nullptr, nullptr, nullptr, split, s, &ex);
  if (rc) return rc;
  rc = colsum_atomic(rows, 32, dz, dbz_scratch, s);
  if (rc) return rc;
  z_wgrad_finish_kernel<<<riqn_cdiv((long)action_space * hidden, 256), 256, 0, s>>>(
      action_space, hidden, dwz_scratch, dbz_scratch, eps_w_zv, eps_b_zv, eps_w_za, eps_b_za, g_mu_zv, g_sig_zv, g_bmu_zv,
      g_bsig_zv, g_mu_za, g_sig_za, g_bmu_za, g_bsig_za);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_argmax_mean(int batch, int num_quantiles, int action_space, const float* q, long long* a_star,
                              void* stream) {
  riqn::note_launches(1);
  if (action_space > 32) return (int)cudaErrorInvalidValue;
  argmax_mean_kernel<<<riqn_cdiv((long)batch * 32, 128), 128, 0, (cudaStream_t)stream>>>(batch, num_quantiles, action_space, q,
                                                                            (int64_t*)a_star);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_iqn_loss_fwd_bwd(int batch, int n_tau, int n_tau_prime, int action_space, const float* q_online,
                                   const float* q_target, const float* tau, const long long* actions,
                                   const long long* a_star, const float* returns, const float* nonterminals,
                                   float gamma_n, float kappa, float* loss, float* dtheta, float* theta_out,
                                   float* target_out, void* stream) {
  riqn::note_launches(1);
  int threads = ((n_tau > n_tau_prime ? n_tau : n_tau_prime) + 31) / 32 * 32;
  if (threads > 1024) threads = 1024;
  if (threads < 32) threads = 32;
  const size_t smem = sizeof(float) * (n_tau_prime + 32);
  iqn_loss_kernel<<<batch, threads, smem, (cudaStream_t)stream>>>(
      batch, n_tau, n_tau_prime, action_space, q_online, q_target, tau, (const int64_t*)actions, (const int64_t*)a_star,
      returns, nonterminals, gamma_n, kappa, loss, dtheta, theta_out, target_out);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_adam_step(long n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int step,
                            float lr, float beta1, float beta2, float eps, float grad_scale, const riqn_dyn_state* dyn,
                            void* stream) {
  riqn::note_launches(1);
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  adam_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(n, params, grads, exp_avg, exp_avg_sq, (float)(-(lr / bc1)),
                                                            (float)sqrt(bc2), eps, beta1, beta2, grad_scale, dyn);
  return (int)cudaGetLastError();
}
