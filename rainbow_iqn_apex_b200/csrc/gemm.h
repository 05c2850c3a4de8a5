// Internal GEMM interface shared by the op implementations (not part of the C-ABI).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace riqn {

// C[m,n] (+)= epi( sum_k A[m*sAm + k*sAk] * B[n*sBn + k*sBk] )
enum Epi {
  EPI_STORE = 0,           // C = alpha*acc
  EPI_BIAS_RELU = 1,       // C = relu(acc + bias[n])
  EPI_BIAS_RELU_NCHW = 2,  // m = b*ohw + p ; C[(b*N + n)*ohw + p] = relu(acc + bias[n])
  EPI_EMBED = 3,           // C = feat[(m / batch)*N + n] * relu(acc + bias[n]), batch = rows per sample (model.py:146-151)
  EPI_ATOMIC = 4,          // C += alpha*acc (atomicAdd; split-K capable)
  EPI_NOISY_WGRAD = 5,     // C += acc ; out2 += acc * eps[m,n]  (dL/dmu, dL/dsigma of NoisyLinear)
  EPI_BIAS = 6,            // C = acc + bias[n]
};

struct EpiArgs {
  const float* bias = nullptr;
  const float* feat = nullptr;
  int batch = 1;
  int ohw = 1;
  float* out2 = nullptr;
  const float* eps = nullptr;
  float alpha = 1.0f;
};

// fp32 CUDA-core GEMM with arbitrary operand strides.  Returns a cudaError_t as int.
int gemm_f32(int M, int N, int K, const float* A, long sAm, long sAk, const float* B, long sBn, long sBk,
             float* C, long ldc, int epi, const EpiArgs& e, int split_k, cudaStream_t stream);

// ---- tcgen05 / TMA path (gemm_tc.cu) ---------------------------------------------------------------------------
enum TcEpi { TC_STORE = 0, TC_BIAS_RELU = 1, TC_ATOMIC = 2, TC_NOISY_WGRAD = 3, TC_BIAS_RELU_NCHW = 4, TC_EMBED = 5,
             TC_COL2IM = 6, TC_CONV = 7, TC_DGRAD = 8 };

struct TcExtra {
  int ohw = 1;
  float alpha = 1.0f;
  const float* feat = nullptr;
  int batch = 1;
  __nv_bfloat16 *o_hi = nullptr, *o_lo = nullptr, *o_hiT = nullptr, *o_loT = nullptr;
  // TC_COL2IM: row m = (b, oh, ow), column n = (c, kh, kw); C is the NCHW image gradient (pad == 0), accumulated into
  int ci_h = 0, ci_w = 0, ci_cin = 0, ci_kh = 0, ci_kw = 0, ci_stride = 0, ci_ow = 0;
  // Strip convolution (TC_CONV): A is the space-to-depth image (B*G*G rows of strip_kc*64 values); k-block kb reads rows
  // m0 + dy*G + dx (shift = kb / strip_kc = dy*strip_t + dx), columns (kb % strip_kc)*64.  Row m = (b, gy, gx) on the
  // G x G grid is a real output iff gy < cv_oh and gx < cv_ow; C is the NCHW fp32 output (relu(acc + bias)); nx_hi / nx_lo
  // (may be null) receive the bf16 images in the NEXT layer's space-to-depth layout (block edge nx_s, grid nx_G).
  int strip_t = 0, strip_G = 0, strip_kc = 0, cv_oh = 0, cv_ow = 0, nx_s = 0, nx_G = 0;
  __nv_bfloat16 *nx_hi = nullptr, *nx_lo = nullptr;
  // Strip-convolution data gradient (TC_DGRAD), the same shifted-row product with negative shifts:
  //   din block row m = (b, gy, gx), column n:   C[m, n] = sum_{shift (dy, dx)} dYg[m - dy*G - dx, :] . Wd[:, shift*N + n]
  // A = dYg (M, dg_cout) K-major (dg_cout <= 64: k-block kb IS shift kb; rows before the first are TMA zero fill),
  // B = Wd (dg_cout, strip_t^2 * N) read MN-major, K = strip_t^2 * 64, strip_G = G.  Column n = (sy, c, sx) (sx fastest)
  // is stored once, without atomics, to the NCHW image C[b, c, gy*s + sy, gx*s + sx] (s = ci_stride, image ci_cin x
  // ci_h x ci_w with G*s <= ci_h, ci_w; pixels beyond G*s, which no output reads, are not written).
  int dg_cout = 0;
  // MN-major operands (mn_major bit 0: A is (K, M) row-major, bit 1: B is (K, N) row-major): the reduction index is the
  // ROW, as in a weight gradient dW = dY^T X taken straight from the row-major activations, or a data gradient
  // dX = dY W read from the untransposed weight (mn_major = 2).  NSPLIT 1 only.
  // wg_t > 0 additionally applies the strip-convolution shifts to B: column n = (shift, within-block) reads the rows
  // k + dy*wg_G + dx of a block matrix with wg_kc*64 columns (shift = n / (wg_kc*64) = dy*wg_t + dx).
  int mn_major = 0, wg_t = 0, wg_G = 0, wg_kc = 0;
  // 16-bit operand formats: 0 = both operand images bf16, 3 = both fp16 (single-pass products only; mixing the two is an
  // illegal instruction), bit 2 = TC_EMBED writes o_hi as fp16(x) and o_lo (optional) as bf16(x) instead of hi / residual
  int fmt = 0;
  // TC_CONV with TWO weight sets over one stacked batch (the online and the target network's trunks over the same frames
  // in one launch): m-tiles [0, grp_mt) use B_hi / B_lo / bias, m-tiles [grp_mt, 2*grp_mt) use b2_hi / b2_lo / bias2.
  // a_wrap != 0: both groups read the SAME A rows (a_rows = rows of the A image; conv1: the pixel block matrix is shared).
  int grp_mt = 0, a_wrap = 0;
  long a_rows = 0;
  const __nv_bfloat16 *b2_hi = nullptr, *b2_lo = nullptr;
  const float* bias2 = nullptr;
};

// C (+)= A B^T, A (M,K) / B (N,K) row-major bf16 (K % 8 == 0); *_lo non-null selects the split-bf16 x3 product.
// (TC_CONV: M = B*G*G grid rows, K = strip_t^2 * strip_kc * 64.)
int gemm_bf16_tc(int M, int N, int K, const __nv_bfloat16* A_hi, const __nv_bfloat16* A_lo, const __nv_bfloat16* B_hi,
                 const __nv_bfloat16* B_lo, float* C, long ldc, int epi, const float* bias, float* out2, const float* eps,
                 int split_k, cudaStream_t s, const TcExtra* ex);
// Split-K factor for a persistent grid of `sms` CTAs: `tiles` output tiles, `kb` reduction blocks of 64.  Minimises
// (rounds of CTAs) x (k-blocks per unit), e.g. 25 tiles -> 11 splits (275 units, two full rounds) rather than 6
// (150 units: a second round for two stragglers).
inline int tc_pick_split(int tiles, long kb, int sms = 148) {
  if (tiles < 1) tiles = 1;
  if (kb < 1) kb = 1;
  long best_cost = -1;
  int best = 1;
  const int smax = (int)(kb < 4L * sms ? kb : 4L * sms);
  for (int s = 1; s <= smax; ++s) {
    const long units = (long)tiles * s, rounds = (units + sms - 1) / sms, per = (kb + s - 1) / s;
    const long cost = rounds * (per + 2);          // +2: fixed per-unit cost (pipeline fill, epilogue)
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = s; }
  }
  return best;
}

int split_bf16(long rows, int cols, const float* src, __nv_bfloat16* hi, __nv_bfloat16* lo, __nv_bfloat16* hiT,
               __nv_bfloat16* loT, cudaStream_t s, int fp16 = 0);

}  // namespace riqn
