// tcgen05 / TMA GEMM for the NoisyLinear hidden layers of the IQN head (the >90% of the learner step's FLOPs:
// reference model.py:153-154 forward, and its dgrad / wgrad), sm_100a only.
//
//   C[m,n] = sum_k A[m,k] * B[n,k]        A (M,K) and B (N,K) both K-major bf16 in HBM, fp32 accumulate in TMEM
//
// * operands arrive by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) into a multi-stage shared-memory ring,
// * one elected thread issues tcgen05.mma.cta_group::1.kind::f16 (UMMA 128x256x16) on shared-memory descriptors,
// * accumulators live in TMEM, double buffered (2 x 256 columns = all 512) so the epilogue of tile i overlaps the
//   MMAs of tile i+1; 4 epilogue warps read them back with tcgen05.ld and apply the fused epilogue,
// * persistent CTAs (one per SM) walk (m-tile, n-tile, k-split) work units round-robin.
//
// Precision: NSPLIT == 1 multiplies bf16(A) * bf16(B).  NSPLIT == 3 takes each operand as hi + lo bf16 pairs
// (a = a_hi + a_lo exactly to ~2^-17) and accumulates a_hi*b_hi + a_hi*b_lo + a_lo*b_hi into the same TMEM
// accumulator: an fp32-faithful product (rel. error ~1e-5 per term) at 3 MMAs per k-step, which keeps the IQN
// loss within 1e-6 of the fp32 reference instead of bf16's 1e-4.
#include <cuda.h>
#include <cudaTypedefs.h>
#include <map>
#include <mutex>
#include <tuple>

#include "common.cuh"
#include "gemm.h"
#include "../../include/riqn_b200.h"

namespace riqn {

using bf16 = __nv_bfloat16;

constexpr int TBM = 128, TBK = 64, UMMA_K = 16;   // tile N (BN) is a template parameter: 256, or 64 / 32 for narrow outputs
// Epilogue warps: a warp may only read the TMEM lane quarter (warp % 4), so they come in sets of four; each set drains an
// equal share of the accumulator columns.  Two sets (8 warps) for the MMA-bound products; FOUR sets for the embedding
// product, whose k = 64 mainloop is over in a microsecond and whose time is all epilogue latency (104 registers per
// thread leave room for 18 warps per SM).
constexpr int epi_warps(int epi) { return epi == TC_EMBED ? 16 : 8; }
constexpr int tc_threads(int epi) { return 64 + 32 * epi_warps(epi); }  // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner


// NSPLIT 1: a_hi*b_hi.  NSPLIT 3: a_hi*b_hi + a_hi*b_lo + a_lo*b_hi.  NSPLIT 2: A is exact in bf16 (e.g. uint8 pixels),
// only B is split: a_hi*b_hi + a_hi*b_lo.
template <int NSPLIT, int BN, int EPI>
struct TcCfg {
  static constexpr int kAOps = NSPLIT == 3 ? 2 : 1, kBOps = NSPLIT == 1 ? 1 : 2;     // hi (+ lo) images per operand
  static constexpr int kOps = kAOps;                                                 // (A images; B tile starts after them)
  static constexpr uint32_t kABytes = TBM * TBK * 2, kBBytes = BN * TBK * 2;
  static constexpr uint32_t kStageBytes = kAOps * kABytes + kBOps * kBBytes;         // 48 / 80 / 96 KB at BN = 256
  static constexpr uint32_t kEpiStage = 32 * 32 * 4;  // per epilogue warp: 32 rows x 32 words for the store transpose
  static constexpr uint32_t kFbBytes = EPI == TC_EMBED ? epi_warps(EPI) * 256 : 0;   // per-warp feat / bias broadcast patches
  static constexpr uint32_t kRingBytes = 224 * 1024 - epi_warps(EPI) * kEpiStage - kFbBytes;   // 192 KB with two warp sets
  static constexpr int kStages = kRingBytes / kStageBytes > 6 ? 6 : kRingBytes / kStageBytes;
  static constexpr uint32_t kTmemCols = 2 * BN < 32 ? 32 : 2 * BN;                   // two accumulator buffers (power of 2)
  static constexpr uint32_t kSmemBytes =
      kStages * kStageBytes + 1024 /*align*/ + epi_warps(EPI) * kEpiStage + 256 /*barriers*/ + kFbBytes;
  static_assert(kSmemBytes <= 232448 && kStages >= 1, "exceeds the 227 KB per-CTA shared memory limit");
};

// ---------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
// TMA store of a staged (rows x 32 elements) 16-bit tile; out-of-range rows / columns are clipped by the tensor map
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(c0), "r"(c1), "r"(src)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"
      "%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128-byte-swizzled operand tile: rows of 64 bf16 (128 B), 8-row swizzle atoms 1024 B apart.
// Descriptor fields (cute/arch/mma_sm100_desc.hpp): start>>4 [0,14), LBO>>4 [16,30) (=1, unused for swizzled
// K-major), SBO>>4 [32,46) (=1024>>4), version=1 [46,48), layout SWIZZLE_128B=2 [61,64).
__device__ __forceinline__ uint64_t umma_desc_k128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}
// MN-major, 128-byte-swizzled operand tile (cute/atom/mma_traits_sm100.hpp, make_umma_desc<Major::MN>): k-rows of 64
// MN-elements (128 B), 8-row swizzle atoms SBO = 1024 B apart along K, further 64-element MN slabs LBO = 8192 B apart.
__device__ __forceinline__ uint64_t umma_desc_mn128(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(8192 >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// kind::f16 instruction descriptor: D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1, K-major both, N>>3 [17,23), M>>4 [24,29)
// (format field: 0 = fp16, 1 = bf16.  The descriptor has separate A / B fields, but a product that MIXES them is an
  // illegal instruction on sm_100a (measured, round 2): both operands must share the format -> fmt is 0 or 3)
__device__ __forceinline__ uint32_t umma_idesc_bf16(int m, int n, int fmt = 0) {
  return (1u << 4) | ((fmt & 1) ? 0u : (1u << 7)) | ((fmt & 2) ? 0u : (1u << 10)) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(m >> 4) << 24);
}
// two floats -> packed 16-bit pair (low half = a), fp16 or bf16
__device__ __forceinline__ uint32_t pack16x2(float a, float b, bool f16) {
  if (f16) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
  }
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// The accumulator arrives with one ROW per lane (tcgen05.ld 32x32b): storing it directly makes every store instruction
// touch 32 different lines with 16-byte pieces (~2 TB/s).  These helpers transpose a 32x32 chunk through a padded
// per-warp shared-memory tile so that each store instruction writes one full row segment (128 B fp32 / 64 B bf16).
// Tile rows are 32 words (128 B) apart and the 16-byte piece j of row r lives at piece slot j ^ (r & 7), so that both the
// deposit (a quarter-warp = 8 rows, same j) and the drain (a quarter-warp = one row, 8 pieces) are bank-conflict free.
// Each lane deposits its row with 8 STS.128; then every instruction moves FOUR rows: lane l handles piece (l & 7) of
// row (l >> 3).
constexpr int kStRow = 32;
// explicit shared-space accesses: the staging pointer comes from an integer-aligned base, which the compiler would
// otherwise treat as a generic address (LD/ST instead of LDS/STS)
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
// st: 32-bit shared address of this warp's 32 x 32-word staging tile
__device__ __forceinline__ void stage_row(uint32_t st, const uint32_t (&w)[32], int lane) {
  __syncwarp();
  const uint32_t row = st + lane * (kStRow * 4);
#pragma unroll
  for (int j = 0; j < 8; ++j) sts128(row + ((j ^ (lane & 7)) << 4), w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
  __syncwarp();
}
__device__ __forceinline__ uint4 staged_piece(uint32_t st, int r, int piece) {
  return lds128(st + r * (kStRow * 4) + ((piece ^ (r & 7)) << 4));
}
__device__ __forceinline__ void warp_store_rows_f32(uint32_t st, const uint32_t (&w)[32], int lane, float* base, long ld,
                                                    int rows_valid) {
  stage_row(st, w, lane);
  const int sub = lane >> 3, piece = lane & 7;
#pragma unroll
  for (int r0 = 0; r0 < 32; r0 += 4) {
    const int r = r0 + sub;
    if (r < rows_valid) *reinterpret_cast<uint4*>(base + (long)r * ld + piece * 4) = staged_piece(st, r, piece);
  }
}
// w[0..15] = hi pairs (cols 2k, 2k+1), w[16..31] = lo pairs: pieces 0-3 go to the hi image, 4-7 to the lo image
__device__ __forceinline__ void warp_store_rows_bf16(uint32_t st, const uint32_t (&w)[32], int lane, bf16* hi_base,
                                                     bf16* lo_base, long ld, int rows_valid) {
  stage_row(st, w, lane);
  const int sub = lane >> 3, piece = lane & 7;
  bf16* dstb = piece < 4 ? hi_base : lo_base;
  if (dstb == nullptr) return;
#pragma unroll
  for (int r0 = 0; r0 < 32; r0 += 4) {
    const int r = r0 + sub;
    if (r < rows_valid) *reinterpret_cast<uint4*>(dstb + (long)r * ld + (piece & 3) * 8) = staged_piece(st, r, piece);
  }
}

// C += alpha * acc (and out2 += alpha * acc * eps for the NoisyLinear weight gradient) on full 128-byte row segments:
// plain 16-byte read-modify-writes when this CTA is the only contributor, red.global.add.v4.f32 under split-K.
template <bool NOISY>
__device__ __forceinline__ void warp_accum_rows_f32(uint32_t st, const uint32_t (&w)[32], int lane, float* c, float* out2,
                                                    const float* eps, long ld, int rows_valid, bool atomic, float alpha) {
  stage_row(st, w, lane);
  const int sub = lane >> 3, piece = lane & 7;
#pragma unroll
  for (int r0 = 0; r0 < 32; r0 += 4) {
    const int r = r0 + sub;
    if (r < rows_valid) {
      const uint4 au = staged_piece(st, r, piece);
      float4 a = make_float4(__uint_as_float(au.x) * alpha, __uint_as_float(au.y) * alpha, __uint_as_float(au.z) * alpha,
                             __uint_as_float(au.w) * alpha);
      const long off = (long)r * ld + piece * 4;
      float4 e = make_float4(0.f, 0.f, 0.f, 0.f);
      if (NOISY) {
        e = *reinterpret_cast<const float4*>(eps + off);
        e.x *= a.x; e.y *= a.y; e.z *= a.z; e.w *= a.w;
      }
      if (!atomic) {
        float4 o = *reinterpret_cast<const float4*>(c + off);
        o.x += a.x; o.y += a.y; o.z += a.z; o.w += a.w;
        *reinterpret_cast<float4*>(c + off) = o;
        if (NOISY) {
          float4 o2 = *reinterpret_cast<const float4*>(out2 + off);
          o2.x += e.x; o2.y += e.y; o2.z += e.z; o2.w += e.w;
          *reinterpret_cast<float4*>(out2 + off) = o2;
        }
      } else {
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(c + off), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w)
                     : "memory");
        if (NOISY)
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(out2 + off), "f"(e.x), "f"(e.y), "f"(e.z),
                       "f"(e.w)
                       : "memory");
      }
    }
  }
}

// Transposed (N, M) bf16 image of a chunk whose 16 words hold the column pairs (2k, 2k+1) of this lane's row: lane pairs
// exchange words so that each lane stores TWO consecutive rows of ONE column (even lanes column 2k, odd lanes 2k+1) --
// 32-bit stores, 64 B contiguous per column.  M must be even.
__device__ __forceinline__ void store_transposed_pairs(bf16* tb, const uint32_t* w16, int n0, int m, int M, int lane,
                                                       bool row_ok) {
  const uint32_t sel = (lane & 1) ? 0x3276u : 0x5410u;
  uint32_t* tp = reinterpret_cast<uint32_t*>(tb + (long)(n0 + (lane & 1)) * M + (m & ~1));
  const long step = M;   // 2 columns = 2*M bf16 = M words
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const uint32_t mine = w16[k];
    const uint32_t other = __shfl_xor_sync(0xffffffffu, mine, 1);
    if (row_ok) tp[(long)k * step] = __byte_perm(mine, other, sel);
  }
}

struct alignas(64) TcArgs {
  CUtensorMap mapO[2];   // TC_EMBED: TMA-store maps of o_hi / o_lo ((M, N) 16-bit row-major, box 32 x 32, 64-byte swizzle)
  int M, N, K;
  int m_tiles, n_tiles, k_splits, kb_per_split, kb_total;
  float* C;
  long ldc;
  const float* bias;     // TC_BIAS_RELU / _NCHW / TC_EMBED
  float* out2;           // TC_NOISY_WGRAD: grad_sigma
  const float* eps;      // TC_NOISY_WGRAD: weight_epsilon (same layout as C)
  float alpha;           // TC_ATOMIC: scale applied to the accumulator
  int vec_acc;           // TC_ATOMIC / TC_NOISY_WGRAD: C (out2, eps) rows are 16-byte aligned -> vectorised accumulate
  int ohw;               // TC_BIAS_RELU_NCHW: m = b*ohw + p -> C[(b*N + n)*ohw + p]
  int ci_h, ci_w, ci_cin, ci_kh, ci_kw, ci_stride, ci_ow;   // TC_COL2IM geometry (pad == 0); TC_DGRAD: image, stride
  const float* feat;     // TC_EMBED: (samples, N) conv features, row m uses feat[m / batch] (batch = rows per sample)
  int batch;
  bf16 *o_hi, *o_lo;     // TC_EMBED: bf16 hi / lo images of the result, row-major (M, N)   (may be null)
  bf16 *o_hiT, *o_loT;   // TC_BIAS_RELU: transposed (N, M) bf16 image of the result          (may be null)
  int strip_t, strip_G, strip_kc, cv_oh, cv_ow, nx_s, nx_G;   // TC_CONV (see gemm.h)
  int mn_major, wg_t, wg_G, wg_kc;                             // MN-major operands / strip weight gradient (gemm.h)
  bf16 *nx_hi, *nx_lo;
  int fmt;               // bit 0: A image is fp16, bit 1: B image is fp16 (else bf16), bit 2: o_hi is written as fp16
  int grp_mt, a_wrap;    // TC_CONV, two weight sets (gemm.h): group 1's B maps live in mapO[0] / mapO[1]
  const float* bias2;
};

template <int NSPLIT, int EPI, int BN>
__global__ void __launch_bounds__(tc_threads(EPI), 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap mapA_hi, const __grid_constant__ CUtensorMap mapA_lo,
               const __grid_constant__ CUtensorMap mapB_hi, const __grid_constant__ CUtensorMap mapB_lo,
               const __grid_constant__ TcArgs p) {
  using Cfg = TcCfg<NSPLIT, BN, EPI>;
  constexpr int TBN = BN;
  constexpr uint32_t TMEM_COLS = Cfg::kTmemCols;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // layout: operand ring | per-warp epilogue staging tiles (4 KB each, 4 KB aligned) | barriers | feat / bias patches
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes + epi_warps(EPI) * Cfg::kEpiStage);
  uint64_t* full = bars;                       // [kStages]  TMA -> MMA
  uint64_t* empty = bars + Cfg::kStages;       // [kStages]  MMA -> TMA
  uint64_t* tfull = bars + 2 * Cfg::kStages;   // [2]        MMA -> epilogue
  uint64_t* tempty = tfull + 2;                // [2]        epilogue -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  const uint32_t epi_stage = (uint32_t)__cvta_generic_to_shared(smem + Cfg::kStages * Cfg::kStageBytes);
  const uint32_t epi_fb = epi_stage + epi_warps(EPI) * Cfg::kEpiStage + 256;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_units = p.m_tiles * p.n_tiles * p.k_splits;

  if (warp == 0 && lane == 0) {
    // descriptor fetch overlaps the barrier / TMEM prologue instead of delaying the first TMA load
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB_hi)) : "memory");
    if (NSPLIT == 3) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA_lo)) : "memory");
    if (NSPLIT >= 2) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB_lo)) : "memory");
    for (int i = 0; i < Cfg::kStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], epi_warps(EPI)); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < total_units; u += gridDim.x) {
        // split-K units are k-split MAJOR: the CTAs in flight walk the SAME reduction range of all output tiles, so each
        // operand slab is fetched from HBM once and shared through L2 (tile-major order read 2.7x the algorithmic bytes)
        const int tiles = p.m_tiles * p.n_tiles;
        const int ks = u / tiles, t = u - ks * tiles;
        const int nt = t % p.n_tiles, mt = t / p.n_tiles;   // n fastest: the A tile is shared by the n-tiles in flight
        const int kb0 = ks * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* s = smem + stage * Cfg::kStageBytes;
          mbar_expect_tx(&full[stage], Cfg::kStageBytes);
          if (EPI == TC_DGRAD) {
            // strip data gradient: k-block kb = shift (dy, dx).  A = dYg rows m0 - dy*G - dx (the first tile's negative
            // rows are zero fill), B = 64 x 64 slabs of the weight image at column kb*N + n, reduction rows 0..63
            const int dy = kb / p.strip_t;
            tma_load_2d(s, &mapA_hi, 0, mt * TBM - dy * p.strip_G - (kb - dy * p.strip_t), &full[stage]);
#pragma unroll
            for (int i = 0; i < TBN / 64; ++i)
              tma_load_2d(s + Cfg::kABytes + i * 8192, &mapB_hi, kb * p.N + nt * TBN + 64 * i, 0, &full[stage]);
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
            continue;
          }
          if (NSPLIT == 1 && p.mn_major) {
            // MN-major operand ((K, MN) row-major): 64 x 64 boxes, inner coordinate = MN offset, outer = reduction row.
            // bit 0: A, bit 1: B; the other operand (if any) stays K-major.
            const int kk = kb * TBK;
            if (p.mn_major & 1) {
#pragma unroll
              for (int i = 0; i < TBM / 64; ++i) tma_load_2d(s + i * 8192, &mapA_hi, mt * TBM + 64 * i, kk, &full[stage]);
            } else {
              tma_load_2d(s, &mapA_hi, kk, mt * TBM, &full[stage]);
            }
            if (p.mn_major & 2) {
#pragma unroll
              for (int i = 0; i < (TBN >= 64 ? TBN / 64 : 1); ++i) {
                int b_in = nt * TBN + 64 * i, b_row = kk;
                if (p.wg_t) {                        // strip weight gradient: this 64-column slab has its own row shift
                  const int slab = b_in >> 6, sft = slab / p.wg_kc, dy = sft / p.wg_t;
                  b_in = (slab - sft * p.wg_kc) << 6;
                  b_row += dy * p.wg_G + (sft - dy * p.wg_t);
                }
                tma_load_2d(s + Cfg::kOps * Cfg::kABytes + i * 8192, &mapB_hi, b_in, b_row, &full[stage]);
              }
            } else {
              tma_load_2d(s + Cfg::kOps * Cfg::kABytes, &mapB_hi, kk, nt * TBN, &full[stage]);
            }
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
            continue;
          }
          int a_col = kb * TBK, a_row = mt * TBM;
          const CUtensorMap *mb_hi = &mapB_hi, *mb_lo = &mapB_lo;
          if (EPI == TC_CONV && p.grp_mt && mt >= p.grp_mt) {   // second weight set (and, for a shared A image, its rows again)
            mb_hi = &p.mapO[0];
            mb_lo = &p.mapO[1];
            if (p.a_wrap) a_row = (mt - p.grp_mt) * TBM;
          }
          if (EPI == TC_CONV) {     // strip convolution: shifted rows of the space-to-depth image
            const int sft = kb / p.strip_kc, dy = sft / p.strip_t;
            a_col = (kb - sft * p.strip_kc) * TBK;
            a_row += dy * p.strip_G + (sft - dy * p.strip_t);
          }
          tma_load_2d(s, &mapA_hi, a_col, a_row, &full[stage]);
          tma_load_2d(s + Cfg::kOps * Cfg::kABytes, mb_hi, kb * TBK, nt * TBN, &full[stage]);
          if (NSPLIT == 3) tma_load_2d(s + Cfg::kABytes, &mapA_lo, a_col, a_row, &full[stage]);
          if (NSPLIT >= 2)
            tma_load_2d(s + Cfg::kAOps * Cfg::kABytes + Cfg::kBBytes, mb_lo, kb * TBK, nt * TBN, &full[stage]);
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (one thread)
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(TBM, TBN, p.fmt);
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++local) {
        const int ks = u / (p.m_tiles * p.n_tiles);
        const int kb0 = ks * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        const int as = local & 1;
        const uint32_t aphase = (local >> 1) & 1;
        mbar_wait(&tempty[as], aphase ^ 1);     // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * TBN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t sb = sa + Cfg::kOps * Cfg::kABytes;
          if (NSPLIT == 1 && (p.mn_major || EPI == TC_DGRAD)) {
            const int mnm = EPI == TC_DGRAD ? 2 : p.mn_major;   // TC_DGRAD: A K-major, B MN-major
            const uint32_t idesc_mn = idesc | ((mnm & 1) ? (1u << 15) : 0u) | ((mnm & 2) ? (1u << 16) : 0u);
#pragma unroll
            for (int k = 0; k < TBK / UMMA_K; ++k) {
              const uint32_t koff_mn = k * (UMMA_K / 8) * 1024;   // MN-major: 16 reduction rows = two 8-row swizzle atoms
              const uint32_t koff_k = k * UMMA_K * 2;             // K-major: bytes inside the 128 B swizzle row
              const uint64_t da = (mnm & 1) ? umma_desc_mn128(sa + koff_mn) : umma_desc_k128(sa + koff_k);
              const uint64_t db = (mnm & 2) ? umma_desc_mn128(sb + koff_mn) : umma_desc_k128(sb + koff_k);
              umma_bf16(tmem_d, da, db, idesc_mn, (kb > kb0 || k > 0) ? 1u : 0u);
            }
            umma_commit(&empty[stage]);
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
            continue;
          }
#pragma unroll
          for (int k = 0; k < TBK / UMMA_K; ++k) {
            const uint32_t koff = k * UMMA_K * 2;   // bytes along K inside the 128 B swizzle row
            const uint64_t a_hi = umma_desc_k128(sa + koff), b_hi = umma_desc_k128(sb + koff);
            umma_bf16(tmem_d, a_hi, b_hi, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            if (NSPLIT >= 2) umma_bf16(tmem_d, a_hi, umma_desc_k128(sb + Cfg::kBBytes + koff), idesc, 1u);
            if (NSPLIT == 3) umma_bf16(tmem_d, umma_desc_k128(sa + Cfg::kABytes + koff), b_hi, idesc, 1u);
          }
          umma_commit(&empty[stage]);             // smem slot free once these MMAs retire
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull[as]);                  // accumulator complete
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (TMEM -> registers -> HBM)
    const int quarter = warp & 3;                 // TMEM lanes [32*quarter, +32) are the ones this warp may read
    const int chalf = (warp - 2) >> 2;            // which half of the accumulator columns this warp drains
    float conv_bias[32];
    if (EPI == TC_CONV) {                         // one n-tile (N <= 64): this warp's 32 columns never change
      constexpr int CH0 = TBN >= 64 ? TBN / 2 : TBN;     // (TC_CONV runs two warp sets)
#pragma unroll
      for (int j = 0; j < 32; ++j) conv_bias[j] = (chalf * CH0 + j < p.N && chalf * CH0 < TBN) ? p.bias[chalf * CH0 + j] : 0.f;
    }
    int local = 0;
    bool conv_grp1 = false;
    for (int u = blockIdx.x; u < total_units; u += gridDim.x, ++local) {
      const int t = u % (p.m_tiles * p.n_tiles);
      const int nt = t % p.n_tiles, mt = t / p.n_tiles;
      if (EPI == TC_CONV && p.grp_mt && (mt >= p.grp_mt) != conv_grp1) {   // a CTA's tiles ascend: this happens at most once
        conv_grp1 = mt >= p.grp_mt;
        constexpr int CH1 = TBN >= 64 ? TBN / 2 : TBN;
        const float* bsrc = conv_grp1 ? p.bias2 : p.bias;
#pragma unroll
        for (int j = 0; j < 32; ++j) conv_bias[j] = (chalf * CH1 + j < p.N && chalf * CH1 < TBN) ? bsrc[chalf * CH1 + j] : 0.f;
      }
      const int as = local & 1;
      const uint32_t aphase = (local >> 1) & 1;
      const int m = mt * TBM + quarter * 32 + lane;
      constexpr int SETS = epi_warps(EPI) / 4;
      constexpr int HALF = TBN >= 32 * SETS ? TBN / SETS : TBN;   // columns per warp set (BN = 32: only the first set has columns)
      // embedding epilogue: lane = row.  The 32 feat / bias values of a chunk are fetched by ONE coalesced load per warp
      // (lane j loads column j) and broadcast through a 256-byte shared-memory patch; the finished 16-bit tiles are staged
      // in the TMA 64-byte-swizzle layout and leave through cp.async.bulk.tensor stores -- no per-thread global stores and
      // no read-back of the staging tile (round 2: the LSU data pipe was the limiter of this kernel)
      const int e_mbase = mt * TBM + quarter * 32;
      const bool e_one_sample = (p.batch & 31) == 0;          // sample-major rows: a warp's 32 rows share one feature row
      const float* embed_feat_row = nullptr;
      if (EPI == TC_EMBED) embed_feat_row = p.feat + (long)((e_mbase < p.M ? e_mbase : 0) / p.batch) * p.N;
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(quarter * 32) << 16) + as * TBN;
#pragma unroll 1
      for (int c = chalf * HALF; c < (chalf + 1) * HALF && c < TBN; c += 32) {
        const int n0 = nt * TBN + c;
        // this chunk's feat / bias values are requested BEFORE the accumulator load: their latency overlaps the TMEM read
        float ef = 0.f, eb = 0.f;
        if (EPI == TC_EMBED && n0 + 32 <= p.N) {
          eb = __ldg(p.bias + n0 + lane);
          if (e_one_sample) ef = __ldg(embed_feat_row + n0 + lane);
        }
        uint32_t v[32];
        tmem_ld32(trow + c, v);
        if (m < p.M && n0 < p.N) {
          if (EPI == TC_STORE || EPI == TC_BIAS_RELU) {
            float* crow = p.C + (long)m * p.ldc + n0;
            if (n0 + 32 <= p.N && (EPI == TC_STORE || (p.M & 1) == 0)) {
              // handled below with the whole warp (coalesced row stores)
            } else if (n0 + 32 <= p.N) {
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                       __uint_as_float(v[j + 3]));
                if (EPI == TC_BIAS_RELU) {
                  const float4 b = *reinterpret_cast<const float4*>(p.bias + n0 + j);
                  o.x = fmaxf(o.x + b.x, 0.f); o.y = fmaxf(o.y + b.y, 0.f);
                  o.z = fmaxf(o.z + b.z, 0.f); o.w = fmaxf(o.w + b.w, 0.f);
                }
                *reinterpret_cast<float4*>(crow + j) = o;
                if (EPI == TC_BIAS_RELU && p.o_hiT) {   // bf16 (N, M) image: lanes = consecutive m -> coalesced
                  p.o_hiT[(long)(n0 + j) * p.M + m] = __float2bfloat16_rn(o.x);
                  p.o_hiT[(long)(n0 + j + 1) * p.M + m] = __float2bfloat16_rn(o.y);
                  p.o_hiT[(long)(n0 + j + 2) * p.M + m] = __float2bfloat16_rn(o.z);
                  p.o_hiT[(long)(n0 + j + 3) * p.M + m] = __float2bfloat16_rn(o.w);
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                if (n0 + j < p.N) {
                  float o = __uint_as_float(v[j]);
                  if (EPI == TC_BIAS_RELU) o = fmaxf(o + p.bias[n0 + j], 0.f);
                  crow[j] = o;
                  if (EPI == TC_BIAS_RELU && p.o_hiT) p.o_hiT[(long)(n0 + j) * p.M + m] = __float2bfloat16_rn(o);
                }
              }
            }
          } else if (EPI == TC_BIAS_RELU_NCHW) {
            const int b = m / p.ohw, pp = m - b * p.ohw;
            float* cb = p.C + ((long)b * p.N + n0) * p.ohw + pp;   // lanes = consecutive pp: coalesced per n
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n0 + j < p.N) cb[(long)j * p.ohw] = fmaxf(__uint_as_float(v[j]) + p.bias[n0 + j], 0.f);
          } else if (EPI == TC_EMBED || EPI == TC_COL2IM || EPI == TC_CONV || EPI == TC_DGRAD) {
            // handled below with the whole warp
          } else if (!(p.vec_acc && n0 + 32 <= p.N)) {
            float* crow = p.C + (long)m * p.ldc + n0;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (n0 + j < p.N) {
                const float o = __uint_as_float(v[j]) * (EPI == TC_ATOMIC ? p.alpha : 1.f);
                if (p.k_splits == 1) {   // sole contributor: += without atomics
                  crow[j] += o;
                  if (EPI == TC_NOISY_WGRAD) p.out2[(long)m * p.ldc + n0 + j] += o * p.eps[(long)m * p.ldc + n0 + j];
                } else {
                  atomicAdd(crow + j, o);
                  if (EPI == TC_NOISY_WGRAD)
                    atomicAdd(p.out2 + (long)m * p.ldc + n0 + j, o * p.eps[(long)m * p.ldc + n0 + j]);
                }
              }
            }
          }
        }
        if (EPI == TC_CONV && n0 < p.N) {
          // strip convolution: relu(acc + bias) -> (optional) fp32 NCHW output + the NEXT layer's space-to-depth images.
          // The bias of this warp's 32 columns sits in registers for the whole kernel (N <= 64 = one n-tile); the image
          // rows go through the staging transpose so that a quarter-warp writes one pixel's 64-byte channel run.
          const int gg = p.strip_G * p.strip_G;
          const int mm = m < p.M ? m : 0;
          const int b = mm / gg, rem = mm - b * gg;
          const int gy = rem / p.strip_G, gx = rem - gy * p.strip_G;
          const bool valid = m < p.M && gy < p.cv_oh && gx < p.cv_ow;
          float x[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = n0 + j < p.N ? fmaxf(__uint_as_float(v[j]) + conv_bias[j], 0.f) : 0.f;
          if (p.C != nullptr && valid) {
            const int plane = p.cv_oh * p.cv_ow;
            float* cb = p.C + ((long)b * p.N + n0) * plane + gy * p.cv_ow + gx;     // lanes = consecutive gx
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (n0 + j < p.N) cb[(long)j * plane] = x[j];
          }
          if (p.nx_hi != nullptr && n0 + 32 <= p.N) {          // warp-uniform
            // this pixel's channels are contiguous in the next layer's space-to-depth row
            long o = -1;
            if (valid) {
              const int sn = p.nx_s, by = gy / sn, bx = gx / sn;
              const long r = ((long)b * p.nx_G + by) * p.nx_G + bx;
              o = r * ((long)sn * sn * p.N) + (long)((gy - by * sn) * sn + (gx - bx * sn)) * p.N + n0;
            }
            uint32_t hw[32];      // [0..15] hi pairs, [16..31] lo pairs
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              const uint32_t hwj = pack16x2(x[j], x[j + 1], false);
              hw[j / 2] = hwj;
              hw[16 + j / 2] = pack16x2(x[j] - __uint_as_float(hwj << 16), x[j + 1] - __uint_as_float(hwj & 0xffff0000u), false);
            }
            const uint32_t st = epi_stage + (warp - 2) * (32 * kStRow * 4);
            stage_row(st, hw, lane);
            const int sub = lane >> 3, piece = lane & 7;
            bf16* dstb = piece < 4 ? p.nx_hi : p.nx_lo;
            uint4 pc[8];                      // all pieces in flight before the first store (one shared-memory latency)
            long orow[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              pc[i] = staged_piece(st, 4 * i + sub, piece);
              orow[i] = __shfl_sync(0xffffffffu, o, 4 * i + sub);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (orow[i] >= 0 && dstb != nullptr) *reinterpret_cast<uint4*>(dstb + orow[i] + (piece & 3) * 8) = pc[i];
          }
        }
        if (EPI == TC_COL2IM && n0 < p.N) {
          // din[b, c, oh*s + kh, ow*s + kw] += dcol[m, (c, kh, kw)]: lane j decodes column n0 + j once, the offsets are
          // broadcast by shuffle; lanes = consecutive output pixels, so one red instruction touches a few lines
          const int khw = p.ci_kh * p.ci_kw;
          const int kcol = n0 + lane;
          int coff = -1;
          if (kcol < p.N) {
            const int c = kcol / khw, r = kcol - c * khw;
            const int kh = r / p.ci_kw, kw = r - kh * p.ci_kw;
            coff = (c * p.ci_h + kh) * p.ci_w + kw;
          }
          const bool row_ok = m < p.M;
          const int mm = row_ok ? m : 0;
          const int b = mm / p.ohw, pp = mm - b * p.ohw;
          const int oh = pp / p.ci_ow, ow = pp - oh * p.ci_ow;
          float* base = p.C + ((long)b * p.ci_cin * p.ci_h + oh * p.ci_stride) * p.ci_w + ow * p.ci_stride;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int off = __shfl_sync(0xffffffffu, coff, j);
            if (row_ok && off >= 0)
              asm volatile("red.global.add.f32 [%0], %1;" ::"l"(base + off), "f"(__uint_as_float(v[j])) : "memory");
          }
        }
        if (EPI == TC_DGRAD && n0 < p.N) {
          // din[b, c, gy*s + sy, gx*s + sx] = acc[m, (sy, c, sx)]: each element exactly once, plain stores.  Lanes are
          // consecutive block columns gx, so one store instruction covers a run of one image row per channel (s = 1: the
          // 32 lanes write 128 contiguous bytes, like the TC_CONV NCHW output); the s = 2 pair (sx = 0, 1) of a channel
          // sits in adjacent columns and leaves as one 8-byte store.  Lane j decodes column n0 + j once; the offsets are
          // broadcast by shuffle.
          const int s = p.ci_stride, sc = s * p.ci_cin;
          const int kcol = n0 + lane;
          int coff = -1;
          if (kcol < p.N) {
            const int sy = kcol / sc, r = kcol - sy * sc, c = r / s;
            coff = (c * p.ci_h + sy) * p.ci_w + (r - c * s);
          }
          const bool row_ok = m < p.M;
          const int gg = p.strip_G * p.strip_G, mm = row_ok ? m : 0;
          const int b = mm / gg, rem = mm - b * gg, gy = rem / p.strip_G, gx = rem - gy * p.strip_G;
          float* base = p.C + ((long)b * p.ci_cin * p.ci_h + gy * s) * p.ci_w + gx * s;
          if (s == 2 && p.vec_acc) {
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              const int off = __shfl_sync(0xffffffffu, coff, j);
              if (row_ok && off >= 0)
                *reinterpret_cast<float2*>(base + off) = make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1]));
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int off = __shfl_sync(0xffffffffu, coff, j);
              if (row_ok && off >= 0) base[off] = __uint_as_float(v[j]);
            }
          }
        }
        if ((EPI == TC_STORE || EPI == TC_EMBED || (EPI == TC_BIAS_RELU && (p.M & 1) == 0) ||
             ((EPI == TC_ATOMIC || EPI == TC_NOISY_WGRAD) && p.vec_acc)) && n0 + 32 <= p.N) {
          const uint32_t st = epi_stage + (warp - 2) * (32 * kStRow * 4);
          const int m_base = mt * TBM + quarter * 32;
          const int rows_valid = min(32, p.M - m_base);            // warp-uniform
          if (rows_valid > 0) {
            if (EPI == TC_STORE) {
              if (p.o_hi != nullptr) {                           // bf16 result (M, N) instead of fp32: 64-byte row pieces
                uint32_t hw2[32];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                  const __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
                  hw2[j] = *reinterpret_cast<const uint32_t*>(&h2);
                  hw2[16 + j] = 0u;
                }
                warp_store_rows_bf16(st, hw2, lane, p.o_hi + (long)m_base * p.N + n0, nullptr, p.N, rows_valid);
              } else {
                warp_store_rows_f32(st, v, lane, p.C + (long)m_base * p.ldc + n0, p.ldc, rows_valid);
              }
            } else if (EPI == TC_ATOMIC) {
              warp_accum_rows_f32<false>(st, v, lane, p.C + (long)m_base * p.ldc + n0, nullptr, nullptr, p.ldc, rows_valid,
                                         p.k_splits > 1, p.alpha);
            } else if (EPI == TC_NOISY_WGRAD) {
              const long o0 = (long)m_base * p.ldc + n0;
              warp_accum_rows_f32<true>(st, v, lane, p.C + o0, p.out2 + o0, p.eps + o0, p.ldc, rows_valid, p.k_splits > 1,
                                        1.f);
            } else if (EPI == TC_BIAS_RELU) {
              const float* br = p.bias + n0;
              uint32_t hw[16];
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 bb = __ldg(reinterpret_cast<const float4*>(br + j));
                const float x0 = fmaxf(__uint_as_float(v[j]) + bb.x, 0.f), x1 = fmaxf(__uint_as_float(v[j + 1]) + bb.y, 0.f);
                const float x2 = fmaxf(__uint_as_float(v[j + 2]) + bb.z, 0.f), x3 = fmaxf(__uint_as_float(v[j + 3]) + bb.w, 0.f);
                const __nv_bfloat162 h01 = __floats2bfloat162_rn(x0, x1), h23 = __floats2bfloat162_rn(x2, x3);
                hw[j / 2] = *reinterpret_cast<const uint32_t*>(&h01);
                hw[j / 2 + 1] = *reinterpret_cast<const uint32_t*>(&h23);
                v[j] = __float_as_uint(x0); v[j + 1] = __float_as_uint(x1);
                v[j + 2] = __float_as_uint(x2); v[j + 3] = __float_as_uint(x3);
              }
              if (p.o_hiT) store_transposed_pairs(p.o_hiT, hw, n0, m, p.M, lane, m < p.M);
              warp_store_rows_f32(st, v, lane, p.C + (long)m_base * p.ldc + n0, p.ldc, rows_valid);
              if (p.o_hi) {                                     // bf16 row-major image (M, N): 64-byte row pieces
                uint32_t hw2[32];
#pragma unroll
                for (int j = 0; j < 16; ++j) { hw2[j] = hw[j]; hw2[16 + j] = 0u; }
                warp_store_rows_bf16(st, hw2, lane, p.o_hi + (long)m_base * p.N + n0, nullptr, p.N, rows_valid);
              }
            } else {
              // x = feat[b] * relu(acc + bias)   (model.py:146-151); N % 32 == 0 is required by the host wrapper.
              const bool f16 = (p.fmt & 4) != 0;
              const uint32_t fb = epi_fb + (warp - 2) * 256;
              const bool row_ok = m < p.M;
              const float* frow = p.feat + (long)((row_ok ? m : 0) / p.batch) * p.N + n0;   // per-row feat (several samples per warp)
              // one image: the two 2 KB halves of the staging tile alternate, so only the store of TWO tiles ago must have
              // read its half (the store of the previous tile stays in flight); two images use both halves every tile
              const bool one_img = p.o_lo == nullptr;
              const uint32_t st0 = one_img ? st + (local & 1) * 2048 : st;
              if (lane == 0) { if (one_img) tma_store_wait_read1(); else tma_store_wait_read(); }
              __syncwarp();
              asm volatile("st.shared.b32 [%0], %1;" ::"r"(fb + lane * 4), "r"(__float_as_uint(ef)) : "memory");
              asm volatile("st.shared.b32 [%0], %1;" ::"r"(fb + 128 + lane * 4), "r"(__float_as_uint(eb)) : "memory");
              __syncwarp();
              uint32_t w0[16], w1[16];                            // image 0 / image 1 column pairs of this lane's row
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const uint4 bu = lds128(fb + 128 + 16 * j);
                uint4 fu;
                if (e_one_sample) fu = lds128(fb + 16 * j);
                else fu = __ldg(reinterpret_cast<const uint4*>(frow) + j);
                const float x0 = __uint_as_float(fu.x) * fmaxf(__uint_as_float(v[4 * j]) + __uint_as_float(bu.x), 0.f);
                const float x1 = __uint_as_float(fu.y) * fmaxf(__uint_as_float(v[4 * j + 1]) + __uint_as_float(bu.y), 0.f);
                const float x2 = __uint_as_float(fu.z) * fmaxf(__uint_as_float(v[4 * j + 2]) + __uint_as_float(bu.z), 0.f);
                const float x3 = __uint_as_float(fu.w) * fmaxf(__uint_as_float(v[4 * j + 3]) + __uint_as_float(bu.w), 0.f);
                if (p.C && row_ok) *reinterpret_cast<float4*>(p.C + (long)m * p.N + n0 + 4 * j) = make_float4(x0, x1, x2, x3);
                if (f16) {            // fp16(x) feeds the single-pass head forward, bf16(x) the backward products
                  w0[2 * j] = pack16x2(x0, x1, true); w0[2 * j + 1] = pack16x2(x2, x3, true);
                  w1[2 * j] = pack16x2(x0, x1, false); w1[2 * j + 1] = pack16x2(x2, x3, false);
                } else {              // bf16 hi + residual lo (split-bf16 x3 head forward)
                  const uint32_t h0 = pack16x2(x0, x1, false), h1 = pack16x2(x2, x3, false);
                  w0[2 * j] = h0; w0[2 * j + 1] = h1;
                  w1[2 * j] = pack16x2(x0 - __uint_as_float(h0 << 16), x1 - __uint_as_float(h0 & 0xffff0000u), false);
                  w1[2 * j + 1] = pack16x2(x2 - __uint_as_float(h1 << 16), x3 - __uint_as_float(h1 & 0xffff0000u), false);
                }
              }
              // 32 rows x 64 bytes per image in the TMA SWIZZLE_64B layout: 16-byte chunk c of row r sits at chunk c ^ ((r >> 1) & 3)
              const uint32_t srow = st0 + lane * 64;
              const int sw = (lane >> 1) & 3;
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                if (p.o_hi) sts128(srow + ((c ^ sw) << 4), w0[4 * c], w0[4 * c + 1], w0[4 * c + 2], w0[4 * c + 3]);
                if (p.o_lo) sts128(srow + 2048 + ((c ^ sw) << 4), w1[4 * c], w1[4 * c + 1], w1[4 * c + 2], w1[4 * c + 3]);
              }
              fence_proxy_async();                                // generic-proxy writes -> visible to the TMA engine
              __syncwarp();
              if (lane == 0) {
                if (p.o_hi) tma_store_2d(&p.mapO[0], st0, n0, m_base);
                if (p.o_lo) tma_store_2d(&p.mapO[1], st0 + 2048, n0, m_base);
                tma_store_commit();
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
    }
  }
  if (EPI == TC_EMBED && warp >= 2 && lane == 0) tma_store_wait_all();   // bulk stores read this CTA's shared memory
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
  }
}

// ---------------------------------------------------------------------------------------------- host side
static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  });
  return fn;
}

// (rows, K) row-major bf16 matrix, box = box_rows x 64 elements, 128-byte swizzle.  Out-of-bounds -> zeros.
static int make_map(CUtensorMap* map, const bf16* base, long rows, long K, int box_rows) {
  auto enc = get_encode();
  if (!enc) return (int)cudaErrorNotSupported;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)(K * sizeof(bf16))};
  cuuint32_t box[2] = {(cuuint32_t)TBK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

// (rows, cols) row-major 16-bit matrix written by TMA stores of 32 x 32 boxes staged in the 64-byte-swizzle layout
static int make_store_map(CUtensorMap* map, const bf16* base, long rows, long cols) {
  auto enc = get_encode();
  if (!enc) return (int)cudaErrorNotSupported;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)(cols * sizeof(bf16))};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

template <int NSPLIT, int EPI, int BN>
static int launch_tc(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo,
                     const TcArgs& p, cudaStream_t s) {
  using Cfg = TcCfg<NSPLIT, BN, EPI>;
  static PerDeviceOnce attr_once;
  const int attr_dev = PerDeviceOnce::device();
  if (!attr_once.done[attr_dev]) {
    RIQN_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<NSPLIT, EPI, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)Cfg::kSmemBytes));
    attr_once.done[attr_dev] = true;
  }
  int sms = attr_once.sms[attr_dev];
  if (!sms) {
    RIQN_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, attr_dev));
    attr_once.sms[attr_dev] = sms;
  }
  const int units = p.m_tiles * p.n_tiles * p.k_splits;
  const int grid = units < sms ? units : sms;
  gemm_tc_kernel<NSPLIT, EPI, BN><<<grid, tc_threads(EPI), Cfg::kSmemBytes, s>>>(a_hi, a_lo, b_hi, b_lo, p);
  return (int)cudaGetLastError();
}

// C (+)= A * B^T on the tensor cores.  A (M,K), B (N,K) bf16 row-major (K % 8 == 0); *_lo may be null (NSPLIT 1).
int gemm_bf16_tc(int M, int N, int K, const bf16* A_hi, const bf16* A_lo, const bf16* B_hi, const bf16* B_lo, float* C,
                 long ldc, int epi, const float* bias, float* out2, const float* eps, int split_k, cudaStream_t s,
                 const TcExtra* ex) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  if ((K % 8) && !(ex != nullptr && ex->mn_major == 3)) return (int)cudaErrorInvalidValue;   // both MN-major: K counts rows
  const bool split3 = A_lo != nullptr && B_lo != nullptr;
  const bool split2 = A_lo == nullptr && B_lo != nullptr;
  // narrow outputs (conv channels, embedding width) get narrow tiles; only the epilogues that occur with them exist
  const bool narrow_ok = epi == TC_BIAS_RELU_NCHW || epi == TC_CONV || ((epi == TC_ATOMIC || epi == TC_STORE) && !split3 && !split2);
  const bool strip = epi == TC_CONV;
  if (strip && (ex == nullptr || ex->strip_t < 1 || ex->strip_kc < 1 || ex->strip_G < 1 || N > 64 ||
                K != ex->strip_t * ex->strip_t * ex->strip_kc * TBK || (ex->nx_hi && (N % 32))))
    return (int)cudaErrorInvalidValue;
  const long a_k = strip ? (long)ex->strip_kc * TBK : K;       // row length of the A image
  const bool mn = ex != nullptr && ex->mn_major != 0;
  if (mn) {
    // A (K, M), B (K, N) row-major; only the plain single-bf16 product with full-width (or 64-wide) N tiles
    if (split3 || split2 || ((ex->mn_major & 1) && (M % 8)) || ((ex->mn_major & 2) && (N % 8)) ||
        (((ex->mn_major & 3) != 3) && (K % 8)))
      return (int)cudaErrorInvalidValue;
  }
  int bn = (ex != nullptr && ex->mn_major) ? ((narrow_ok && N <= 64) ? 64 : 256)
                                           : (narrow_ok && N <= 32) ? 32 : (narrow_ok && N <= 64) ? 64 : 256;
  if (epi == TC_BIAS_RELU && split3 && !(ex != nullptr && ex->mn_major) && N % 128 == 0) {
    // head forward with few rows (K = 32 quantiles): 128-wide tiles when they fill the persistent grid's last round
    // noticeably better (512 tiles = 3.46 rounds of 148 CTAs -> 1024 half tiles = 6.92 rounds)
    const long mt = (M + TBM - 1) / TBM, t256 = mt * ((N + 255) / 256), t128 = mt * (N / 128);
    auto eff = [](long t) { const long r = (t + 147) / 148; return (double)t / (double)(r * 148); };
    if (eff(t128) > eff(t256) + 0.08) bn = 128;
  }
  if (epi == TC_EMBED) bn = 128;   // four epilogue warp sets x one 32-column chunk; 64 KB stages leave room for their staging
  // (32-wide tiles for conv3's 324 strip tiles were tried: slower -- only four epilogue warps drain a 32-column tile)
  const bool dgrad = epi == TC_DGRAD;
  if (dgrad) {
    if (ex == nullptr || split3 || split2 || mn || ex->strip_t < 1 || ex->strip_G < 1 || ex->dg_cout < 8 || ex->dg_cout > 64 ||
        ex->dg_cout % 8 || K != ex->strip_t * ex->strip_t * TBK || ex->ci_stride < 1 || ex->ci_cin < 1 ||
        N != ex->ci_stride * ex->ci_stride * ex->ci_cin || N % 8 || M % (ex->strip_G * ex->strip_G) ||
        ex->strip_G * ex->ci_stride > ex->ci_h || ex->strip_G * ex->ci_stride > ex->ci_w)
      return (int)cudaErrorInvalidValue;
    bn = N <= 64 ? 64 : N <= 128 ? 128 : 256;    // conv3: 64 columns, conv2: 128 -- one n-tile either way
  }
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  int rc;
  if (dgrad) {
    rc = make_map(&ma_hi, A_hi, M, ex->dg_cout, TBM);                                    // dYg (M, Cout)
    if (rc) return rc;
    rc = make_map(&mb_hi, B_hi, ex->dg_cout, (long)ex->strip_t * ex->strip_t * N, 64);   // Wd (Cout, t*t*N)
    if (rc) return rc;
  } else if (mn) {
    const long b_cols = ex->wg_t ? (long)ex->wg_kc * TBK : N;      // strip weight gradient: B is the block matrix
    rc = (ex->mn_major & 1) ? make_map(&ma_hi, A_hi, K, M, 64) : make_map(&ma_hi, A_hi, M, K, TBM);
    if (rc) return rc;
    rc = (ex->mn_major & 2) ? make_map(&mb_hi, B_hi, K, b_cols, 64) : make_map(&mb_hi, B_hi, N, K, bn);
    if (rc) return rc;
  } else {
    rc = make_map(&ma_hi, A_hi, (ex && ex->a_rows) ? ex->a_rows : M, a_k, TBM);
    if (rc) return rc;
    rc = make_map(&mb_hi, B_hi, N, K, bn);
    if (rc) return rc;
  }
  ma_lo = ma_hi;
  mb_lo = mb_hi;
  if (split3) {
    rc = make_map(&ma_lo, A_lo, (ex && ex->a_rows) ? ex->a_rows : M, a_k, TBM);
    if (rc) return rc;
  }
  if (split3 || split2) {
    rc = make_map(&mb_lo, B_lo, N, K, bn);
    if (rc) return rc;
  }
  TcArgs p;
  p.M = M; p.N = N; p.K = K;
  p.m_tiles = (M + TBM - 1) / TBM;
  p.n_tiles = (N + bn - 1) / bn;
  p.kb_total = (K + TBK - 1) / TBK;
  if (split_k < 1) split_k = 1;
  if (split_k > p.kb_total) split_k = p.kb_total;
  p.kb_per_split = (p.kb_total + split_k - 1) / split_k;
  p.k_splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  if (p.k_splits > 1 && epi != TC_ATOMIC && epi != TC_NOISY_WGRAD) return (int)cudaErrorInvalidValue;
  p.C = C; p.ldc = ldc; p.bias = bias; p.out2 = out2; p.eps = eps;
  p.alpha = ex ? ex->alpha : 1.f;
  p.vec_acc = (ldc % 4 == 0) && (reinterpret_cast<uintptr_t>(C) & 15) == 0 && (reinterpret_cast<uintptr_t>(out2) & 15) == 0 &&
              (reinterpret_cast<uintptr_t>(eps) & 15) == 0;
  p.ohw = ex ? ex->ohw : 1; p.feat = ex ? ex->feat : nullptr; p.batch = ex ? ex->batch : 1;
  p.ci_h = ex ? ex->ci_h : 0; p.ci_w = ex ? ex->ci_w : 0; p.ci_cin = ex ? ex->ci_cin : 0; p.ci_kh = ex ? ex->ci_kh : 0;
  p.ci_kw = ex ? ex->ci_kw : 0; p.ci_stride = ex ? ex->ci_stride : 0; p.ci_ow = ex ? ex->ci_ow : 0;
  p.strip_t = ex ? ex->strip_t : 0; p.strip_G = ex ? ex->strip_G : 0; p.strip_kc = ex ? ex->strip_kc : 0;
  p.cv_oh = ex ? ex->cv_oh : 0; p.cv_ow = ex ? ex->cv_ow : 0; p.nx_s = ex ? ex->nx_s : 0; p.nx_G = ex ? ex->nx_G : 0;
  p.nx_hi = ex ? ex->nx_hi : nullptr; p.nx_lo = ex ? ex->nx_lo : nullptr;
  p.mn_major = mn ? ex->mn_major : 0; p.wg_t = ex ? ex->wg_t : 0; p.wg_G = ex ? ex->wg_G : 0; p.wg_kc = ex ? ex->wg_kc : 0;
  if (epi == TC_COL2IM && (ex == nullptr || p.ci_kh * p.ci_kw * p.ci_cin != N || split3 || split2)) return (int)cudaErrorInvalidValue;
  if (dgrad) p.vec_acc = (reinterpret_cast<uintptr_t>(C) & 7) == 0 && (p.ci_w & 1) == 0;   // s = 2: 8-byte pair stores
  p.o_hi = ex ? ex->o_hi : nullptr; p.o_lo = ex ? ex->o_lo : nullptr;
  p.o_hiT = ex ? ex->o_hiT : nullptr; p.o_loT = ex ? ex->o_loT : nullptr;
  p.fmt = ex ? ex->fmt : 0;
  p.grp_mt = ex ? ex->grp_mt : 0; p.a_wrap = ex ? ex->a_wrap : 0; p.bias2 = ex ? ex->bias2 : nullptr;
  if (p.grp_mt) {
    if (epi != TC_CONV || !ex->b2_hi || !ex->bias2 || p.m_tiles != 2 * p.grp_mt || (split3 || split2) != (ex->b2_lo != nullptr))
      return (int)cudaErrorInvalidValue;
    if ((rc = make_map(&p.mapO[0], ex->b2_hi, N, K, bn))) return rc;
    p.mapO[1] = p.mapO[0];
    if (ex->b2_lo && (rc = make_map(&p.mapO[1], ex->b2_lo, N, K, bn))) return rc;
  }
  if ((p.fmt & 3) && (split3 || split2)) return (int)cudaErrorInvalidValue;      // fp16 images are single-pass operands
  if ((p.fmt & 3) == 1 || (p.fmt & 3) == 2) return (int)cudaErrorInvalidValue;   // mixed fp16 x bf16: illegal instruction
  if ((p.fmt & 4) && epi != TC_EMBED) return (int)cudaErrorInvalidValue;
  if (epi == TC_EMBED && ((N % 32) || (M % 2) || p.o_hiT || p.o_loT)) return (int)cudaErrorInvalidValue;
  if (epi == TC_EMBED) {            // the 16-bit images leave through TMA stores
    if (p.o_hi && (rc = make_store_map(&p.mapO[0], p.o_hi, M, N))) return rc;
    if (p.o_lo && (rc = make_store_map(&p.mapO[1], p.o_lo, M, N))) return rc;
  }
#define RIQN_TC_GO(NS, EP) return launch_tc<NS, EP, 256>(ma_hi, ma_lo, mb_hi, mb_lo, p, s)
#define RIQN_TC_NARROW(NS, EP)                                                                  \
  if (bn == 32) return launch_tc<NS, EP, 32>(ma_hi, ma_lo, mb_hi, mb_lo, p, s);                  \
  if (bn == 64) return launch_tc<NS, EP, 64>(ma_hi, ma_lo, mb_hi, mb_lo, p, s)
  if (split3) {
    switch (epi) {
      case TC_STORE: RIQN_TC_GO(3, TC_STORE);
      case TC_BIAS_RELU:
        if (bn == 128) return launch_tc<3, TC_BIAS_RELU, 128>(ma_hi, ma_lo, mb_hi, mb_lo, p, s);
        RIQN_TC_GO(3, TC_BIAS_RELU);
      case TC_ATOMIC: RIQN_TC_GO(3, TC_ATOMIC);
      case TC_NOISY_WGRAD: RIQN_TC_GO(3, TC_NOISY_WGRAD);
      case TC_BIAS_RELU_NCHW: RIQN_TC_NARROW(3, TC_BIAS_RELU_NCHW); RIQN_TC_GO(3, TC_BIAS_RELU_NCHW);
      case TC_CONV: RIQN_TC_NARROW(3, TC_CONV); break;
      case TC_EMBED: return launch_tc<3, TC_EMBED, 128>(ma_hi, ma_lo, mb_hi, mb_lo, p, s);
    }
  } else if (split2) {
    switch (epi) {
      case TC_BIAS_RELU_NCHW: RIQN_TC_NARROW(2, TC_BIAS_RELU_NCHW); RIQN_TC_GO(2, TC_BIAS_RELU_NCHW);
      case TC_CONV: RIQN_TC_NARROW(2, TC_CONV); break;
      case TC_STORE: RIQN_TC_GO(2, TC_STORE);
      default: return (int)cudaErrorInvalidValue;
    }
  } else {
    switch (epi) {
      case TC_STORE: RIQN_TC_NARROW(1, TC_STORE); RIQN_TC_GO(1, TC_STORE);
      case TC_COL2IM: RIQN_TC_GO(1, TC_COL2IM);
      case TC_DGRAD:
        if (bn == 64) return launch_tc<1, TC_DGRAD, 64>(ma_hi, ma_lo, mb_hi, mb_lo, p, s);
        if (bn == 128) return launch_tc<1, TC_DGRAD, 128>(ma_hi, ma_lo, mb_hi, mb_lo, p, s);
        RIQN_TC_GO(1, TC_DGRAD);
      case TC_BIAS_RELU: RIQN_TC_GO(1, TC_BIAS_RELU);
      case TC_ATOMIC: RIQN_TC_NARROW(1, TC_ATOMIC); RIQN_TC_GO(1, TC_ATOMIC);
      case TC_NOISY_WGRAD: RIQN_TC_GO(1, TC_NOISY_WGRAD);
      case TC_BIAS_RELU_NCHW: RIQN_TC_NARROW(1, TC_BIAS_RELU_NCHW); RIQN_TC_GO(1, TC_BIAS_RELU_NCHW);
      case TC_CONV: RIQN_TC_NARROW(1, TC_CONV); break;
      case TC_EMBED: return launch_tc<1, TC_EMBED, 128>(ma_hi, ma_lo, mb_hi, mb_lo, p, s);
    }
  }
#undef RIQN_TC_NARROW
#undef RIQN_TC_GO
  return (int)cudaErrorInvalidValue;
}

// ---------------------------------------------------------------------------------------------- operand producers
// fp32 (rows, cols) -> bf16 hi (+ lo = bf16(x - hi)), optionally also transposed copies (cols, rows).
__global__ void split_bf16_kernel(long rows, int cols, const float* __restrict__ src, bf16* __restrict__ hi,
                                  bf16* __restrict__ lo, bf16* __restrict__ hiT, bf16* __restrict__ loT, int fp16) {
  __shared__ float tile[32][33];
  const long r0 = (long)blockIdx.y * 32;
  const int c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const long r = r0 + i;
    const int c = c0 + tx;
    float x = 0.f;
    if (r < rows && c < cols) {
      x = src[r * cols + c];
      if (fp16) {                       // hi = fp16(x); lo (optional) = bf16(x), NOT a residual
        reinterpret_cast<__half*>(hi)[r * cols + c] = __float2half_rn(x);
        if (lo) lo[r * cols + c] = __float2bfloat16_rn(x);
        continue;
      }
      const bf16 h = __float2bfloat16_rn(x);
      if (hi) hi[r * cols + c] = h;
      if (lo) lo[r * cols + c] = __float2bfloat16_rn(x - __bfloat162float(h));
    }
    tile[i][tx] = x;
  }
  if (!hiT) return;
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i;
    const long r = r0 + tx;
    if (r < rows && c < cols) {
      const float x = tile[tx][i];
      const bf16 h = __float2bfloat16_rn(x);
      hiT[(long)c * rows + r] = h;
      if (loT) loT[(long)c * rows + r] = __float2bfloat16_rn(x - __bfloat162float(h));
    }
  }
}

int split_bf16(long rows, int cols, const float* src, bf16* hi, bf16* lo, bf16* hiT, bf16* loT, cudaStream_t s, int fp16) {
  if (fp16 && (hi == nullptr || hiT != nullptr || loT != nullptr)) return (int)cudaErrorInvalidValue;
  dim3 grid((cols + 31) / 32, (unsigned)((rows + 31) / 32));
  split_bf16_kernel<<<grid, 256, 0, s>>>(rows, cols, src, hi, lo, hiT, loT, fp16);
  return (int)cudaGetLastError();
}

}  // namespace riqn

using namespace riqn;

__global__ void split_bf16_scaled_kernel(long n, const float* __restrict__ src, float scale, riqn::bf16* __restrict__ hi,
                                         riqn::bf16* __restrict__ lo) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = __fdiv_rn(src[i], scale);      // weight / 255, like the reference divides the pixel
  const riqn::bf16 h = __float2bfloat16_rn(x);
  hi[i] = h;
  if (lo) lo[i] = __float2bfloat16_rn(x - __bfloat162float(h));
}

RIQN_API int riqn_split_bf16_scaled(long rows, int cols, const float* src, float scale, void* hi, void* lo, void* stream) {
  riqn::note_launches(1);
  const long n = rows * cols;
  split_bf16_scaled_kernel<<<riqn_cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(n, src, scale, (riqn::bf16*)hi, (riqn::bf16*)lo);
  return (int)cudaGetLastError();
}

struct SplitJobs {
  riqn_split_job j[12];
  int blk_end[12];
  int n;
};

__global__ void split_bf16_multi_kernel(SplitJobs t) {
  int ji = 0;
  while (ji < t.n - 1 && (int)blockIdx.x >= t.blk_end[ji]) ++ji;
  const riqn_split_job& J = t.j[ji];
  const int idx = (blockIdx.x - (ji ? t.blk_end[ji - 1] : 0)) * blockDim.x + threadIdx.x;
  if (idx >= J.rows * J.cols) return;
  const int r = idx / J.cols, c = idx - r * J.cols;
  float x = J.src[(long)r * J.cols + (J.perm ? J.perm[c] : c)];
  if (J.div != 1.0f) x = __fdiv_rn(x, J.div);
  const riqn::bf16 h = __float2bfloat16_rn(x);
  reinterpret_cast<riqn::bf16*>(J.hi)[idx] = h;
  if (J.lo) reinterpret_cast<riqn::bf16*>(J.lo)[idx] = __float2bfloat16_rn(x - __bfloat162float(h));
  if (J.hi_t) reinterpret_cast<riqn::bf16*>(J.hi_t)[(long)c * J.rows + r] = h;
}

RIQN_API int riqn_split_bf16_multi(int n_jobs, const riqn_split_job* jobs, void* stream) {
  riqn::note_launches(1);
  if (n_jobs < 1 || n_jobs > 12 || jobs == nullptr) return (int)cudaErrorInvalidValue;
  SplitJobs t;
  t.n = n_jobs;
  int blocks = 0;
  for (int i = 0; i < n_jobs; ++i) {
    if (jobs[i].src == nullptr || jobs[i].hi == nullptr || jobs[i].rows < 1 || jobs[i].cols < 1) return (int)cudaErrorInvalidValue;
    t.j[i] = jobs[i];
    blocks += (int)riqn_cdiv((long)jobs[i].rows * jobs[i].cols, 256);
    t.blk_end[i] = blocks;
  }
  split_bf16_multi_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(t);
  return (int)cudaGetLastError();
}

RIQN_API int riqn_split_bf16(long rows, int cols, const float* src, void* hi, void* lo, void* hi_t, void* lo_t, int fp16,
                             void* stream) {
  riqn::note_launches(1);
  return split_bf16(rows, cols, src, (bf16*)hi, (bf16*)lo, (bf16*)hi_t, (bf16*)lo_t, (cudaStream_t)stream, fp16);
}

RIQN_API int riqn_gemm_bf16_tc(int M, int N, int K, const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                               float* c, long ldc, int epilogue, const float* bias, float* out2, const float* eps,
                               int split_k, void* c_t_bf16, void* c_bf16, int fmt, void* stream) {
  riqn::note_launches(1);
  TcExtra ex;
  ex.o_hiT = (bf16*)c_t_bf16;
  ex.o_hi = (bf16*)c_bf16;
  ex.fmt = fmt & 3;
  if (c_bf16 && (epilogue != TC_BIAS_RELU || (M & 1) || (N % 32))) return (int)cudaErrorInvalidValue;
  return gemm_bf16_tc(M, N, K, (const bf16*)a_hi, (const bf16*)a_lo, (const bf16*)b_hi, (const bf16*)b_lo, c, ldc, epilogue,
                      bias, out2, eps, split_k, (cudaStream_t)stream, &ex);
}

RIQN_API int riqn_gemm_bf16_tc_mn(int M, int N, int K, const void* a, const void* b_kn, int a_is_km, float* c, long ldc,
                                  int epilogue, float* out2, const float* eps, float alpha, int split_k, void* c_bf16,
                                  int fmt, void* stream) {
  riqn::note_launches(1);
  if (epilogue != TC_STORE && epilogue != TC_ATOMIC && epilogue != TC_NOISY_WGRAD) return (int)cudaErrorInvalidValue;
  if (c_bf16 && (epilogue != TC_STORE || (N % 32))) return (int)cudaErrorInvalidValue;
  TcExtra ex;
  ex.o_hi = (bf16*)c_bf16;
  ex.mn_major = a_is_km ? 3 : 2;
  ex.alpha = alpha;
  ex.fmt = fmt & 3;
  return gemm_bf16_tc(M, N, K, (const bf16*)a, nullptr, (const bf16*)b_kn, nullptr, c, ldc, epilogue, nullptr, out2, eps,
                      split_k, (cudaStream_t)stream, &ex);
}
