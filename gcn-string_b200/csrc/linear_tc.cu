// K1 / K9 on the 5th-generation tensor cores: fp32-accurate dense transforms for widths that
// are multiples of 128, as 3xTF32 error-compensated products issued with tcgen05.mma.
//
//   C[M, N] (+)= A[M, K] . B[K, N] (+ bias)        A: activations (fp32, any leading dim)
//                                                   B: weights, pre-split once per call
// fp32 parity (BASELINE.json: 1e-5 relative) rules out a single TF32/BF16 pass (~1e-3).  Each
// operand is split a = a_hi + a_lo with a_hi = tf32(a) rounded to nearest, a_lo = a - a_hi, and
//   A.B ~= A_hi.B_hi + A_hi.B_lo + A_lo.B_hi      (the dropped A_lo.B_lo term is ~2^-22)
// accumulates in fp32 in tensor memory: three kind::tf32 products per K step.
//
// The tensor core adds each K=8 step into the fp32 accumulator with TRUNCATION, a bias that grows
// with the number of steps of a chain (~n * 2^-26).  So the main term A_hi.B_hi and the 2^-11-smaller
// correction terms accumulate in SEPARATE tensor-memory accumulators that meet in fp32 adds in the
// epilogue, and chains are kept short: forward / dX reductions longer than 768 are chunked (launch()),
// the weight gradient folds its chains into a running fp32 sum every 16 K blocks.
//
// Two kernels (profiles/r01_gemm_kernels.md has the measurement behind every structural choice):
//   linear_tc_pair_kernel   forward and input gradient: persistent CTA pairs (cta_group::2), A operand
//                           split by converter warps straight into TENSOR MEMORY (TS-mode MMA), weight
//                           tiles split across the pair, TMA-store / reduce-add epilogue
//   linear_f16_pass256_kernel  its fp16 form for output widths that are multiples of 256: 256 columns per pass, the
//                           split A operand in shared memory (SS-mode MMA), one fetch and split of A per pass
//   wgrad_tc_kernel         weight gradient: reduction over the rows, A^T gathered into tensor memory,
//                           dH split in shared memory as an MN-major operand
#include <cuda.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "prep.cuh"

namespace gcs {
namespace tc {

constexpr int BM = 128, BN = 128, BK = 32;
constexpr int kStages = 4;    // shared-memory stages (TMA)
constexpr int kWgAStages = 2; // ... of the weight-gradient kernel (it also keeps a running sum in TMEM)
constexpr int kConvWarps = 8; // converter warps: two per TMEM lane quarter, 16 of the 32 K columns each
constexpr int kThreads = 64 + 32 * kConvWarps;
constexpr uint32_t A_RAW_BYTES = BM * BK * 4;          // 16 KB
constexpr uint32_t ACC_MAIN = 0, ACC_CORR = 128, A_COL = 256, kTmemCols = 512;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem desc], kind::tf32
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// 1 in exactly one lane of the (converged) warp
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred;
}
__device__ __forceinline__ uint32_t rna_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// In-kernel operand split.  ptxas expands cvt.rna.tf32 into ~6 integer/predicate instructions, which made the
// converter warps' per-K-block chain (~1090 clk) the bound of the mainloop.  Round-to-nearest (ties away, as rna)
// on the raw bits is two integer instructions; the low part is handed over unrounded - the tensor core ignores the
// 13 low mantissa bits of a tf32 operand, i.e. truncates it (|lo| <= 2^-11 |x|, so that costs <= 2^-21 |x|).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xFFFFE000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

#define GCS_R32(v) v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8], v[9], v[10], v[11], v[12], v[13], v[14], v[15], \
                   v[16], v[17], v[18], v[19], v[20], v[21], v[22], v[23], v[24], v[25], v[26], v[27], v[28], v[29], v[30], v[31]

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31]) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
}

// Shared-memory matrix descriptor, K-major, SWIZZLE_128B, 128 B rows: 8-row atoms 1024 B apart.
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);         // start address, 16 B units
  d |= static_cast<uint64_t>(0) << 16;                            // leading byte offset (unused: one atom along K)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                    // stride byte offset between 8-row atoms
  d |= static_cast<uint64_t>(1) << 46;                            // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                            // SWIZZLE_128B
  return d;
}

// ---------------------------------------------------------------------------------------------
// Forward / dX kernel: persistent CTA pairs (tcgen05 cta_group::2).
//
// ncu on the one-CTA-per-tile kernel this replaced (profiles/r01_gemm_kernels.md): 12.7 GB of TMA loads per
// launch at 9.3 TB/s = the ~42 B/clk/SM the L2 -> SM fabric delivers; the tensor pipe waits for
// the weight tiles, which every CTA streams in full (32 KB of the 48 KB per K block).  A CTA pair
// computes a 256 x 128 tile with ONE copy of the weight tiles split across the two SMs: each CTA
// loads its own 128 rows of A (16 KB) and only HALF of the weight rows (64 of B_hi and 64 of B_lo,
// 16 KB), so the ingest per SM and K block drops from 48 KB to 32 KB for the same tensor work.
//
// Per CTA and stage the shared tile is [A raw 128 x 32 | B_hi half 64 x 32 | B_lo half 64 x 32];
// the two weight halves are adjacent, so the pair-wide B operand of
//     MMA1:  A_hi . [B_hi(0:64) ; B_lo(0:64) | B_hi(64:128) ; B_lo(64:128)]     N = 256
// is one 128-row K-major operand per CTA, and
//     MMA2:  A_lo . [B_hi(0:64) | B_hi(64:128)]                                 N = 128
// reuses the first 64 rows of it.  Accumulator columns (each CTA, its own 128 rows):
//     [0,64) main n<64 | [64,128) A_hi.B_lo n<64 | [128,192) main n>=64 | [192,256) A_hi.B_lo n>=64
//     [256,384) A_lo.B_hi | [384,512) two tensor-memory stages of the split A operand.
// The leader CTA issues every MMA; the converters of BOTH CTAs arrive on the leader's a_ready
// barrier (remote mbarrier arrive), tcgen05.commit multicasts the "consumed" signals to both CTAs.
constexpr int kPStages = 5;
constexpr int kPAStages = 2;
constexpr uint32_t P_B_BYTES = 64 * BK * 4;              // 8 KB per weight half
constexpr uint32_t P_STAGE_BYTES = A_RAW_BYTES + 2 * P_B_BYTES;   // 32 KB
constexpr uint32_t P_OUT_BYTES = 32 * 32 * 4;            // per converter warp: one 32 x 32 output box staged for the TMA store
constexpr uint32_t kPSmemBytes = kPStages * P_STAGE_BYTES + kConvWarps * P_OUT_BYTES + 1024 + 256;
// fp16 variant (see linear_tc_pair_kernel<true>): K blocks of 64 - two raw fp32 A boxes (32 KB) and the two weight
// halves as fp16 [64 x 64] (8 KB each, 128 B rows like the tf32 tiles) - four stages.
// Converting 64 K elements per row costs ~3x the instructions of the tf32 split of 32 while the tensor time per K block
// stays the same, so the fp16 variant runs SIXTEEN converter warps (four per tensor-memory lane quarter, 16 K elements
// each; 576 threads, <= 112 registers: the epilogue reads its 32 x 32 box in two halves) and three 48 KB stages.
constexpr int kHStages = 3;
constexpr int BKH = 64;
constexpr int kHConvWarps = 16;
constexpr int kHThreads = 64 + 32 * kHConvWarps;
constexpr uint32_t H_STAGE_BYTES = 2 * A_RAW_BYTES + 2 * P_B_BYTES;   // 48 KB
constexpr uint32_t kHSmemBytes = kHStages * H_STAGE_BYTES + kHConvWarps * P_OUT_BYTES + 1024 + 256;
static_assert(kHSmemBytes <= 232448, "fp16 pair kernel exceeds the 227 KB of shared memory per CTA");
constexpr uint32_t P_ACC1 = 0, P_ACC2 = 256, P_A_COL = 384;
// M = 256 across the pair; N = 256 / 128
constexpr uint32_t kPairDesc256 = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(256 >> 3) << 17) |
                                  (static_cast<uint32_t>(256 >> 4) << 24);
constexpr uint32_t kPairDesc128 = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(128 >> 3) << 17) |
                                  (static_cast<uint32_t>(256 >> 4) << 24);
// the same shapes for kind::f16 with F16 operands (format 0) and an F32 accumulator
constexpr uint32_t kPairDesc256H = (1u << 4) | (static_cast<uint32_t>(256 >> 3) << 17) | (static_cast<uint32_t>(256 >> 4) << 24);
constexpr uint32_t kPairDesc128H = (1u << 4) | (static_cast<uint32_t>(128 >> 3) << 17) | (static_cast<uint32_t>(256 >> 4) << 24);

__device__ __forceinline__ void mma_tf32_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_f16_ts_pair(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// fp16 operand split of two neighbouring K elements (already multiplied by the operand's power-of-two scale):
// hi = fp16(y), lo = fp16((y - hi) * 2^11) - both parts carry 11 significant bits in fp16's range, the pair 22 bits
// like the tf32 split; element 2i sits in the low half of the 32-bit tensor-memory cell.
__device__ __forceinline__ void split_f16x2(float y0, float y1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(y0, y1);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn((y0 - hf.x) * 2048.f, (y1 - hf.y) * 2048.f);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// Power-of-two scale that brings an operand with the given |max| to [2^13, 2^14) (fp16 overflows at 65504); 1 for an
// all-zero or non-finite maximum.
__device__ __forceinline__ float f16_scale(float amax) {
  const uint32_t e = (__float_as_uint(amax) >> 23) & 0xFFu;
  if (e == 0u || e == 0xFFu) return 1.f;
  int se = 127 + 13 - (static_cast<int>(e) - 127);
  se = se < 1 ? 1 : (se > 254 ? 254 : se);
  return __uint_as_float(static_cast<uint32_t>(se) << 23);
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(static_cast<uint16_t>(3)) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAITC_%=:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONEC_%=;\n\t"
      "bra WAITC_%=;\n\t"
      "DONEC_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {      // arrive on CTA 0's copy of `bar`
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(bar), "r"(0));
  // default semantics (release at CTA scope) as CUTLASS's ClusterBarrier::arrive(cta_id): a .release.cluster arrive compiles to
  // MEMBAR.ALL.GPU + CCTL.IVALL per arrival (measured: 2100 clk per K block, independent of the tensor work).  What the
  // leader must observe is ordered without it: the TMEM writes by tcgen05.wait::st + fence::before_thread_sync, the
  // TMA-written shared tiles never pass through the generic proxy.
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}

// kF16 = true: the same pipeline on kind::f16 MMAs (K = 16 per instruction at the K = 8 tf32 rate, i.e. half the tensor
// time per product).  Operands are split into fp16 hi + 2^11-scaled fp16 lo (22 bits, as the tf32 split); fp16's narrow
// exponent range is handled by a power-of-two scale per operand: A is multiplied by f16_scale(*a_amax) in the converters
// (a_amax = running |max| of the tensor, maintained by its producer kernels), the weights by b_scale in the split
// kernel; the epilogue undoes both.  Elements more than 2^28 below the operand's maximum lose relative precision -
// an absolute error of 2^-36 of the maximum, far below fp32 rounding of the sums they enter.
template <bool kF16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kF16 ? kHThreads : kThreads, 1) linear_tc_pair_kernel(
    const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b_hi,
    const __grid_constant__ CUtensorMap map_b_lo, const __grid_constant__ CUtensorMap map_c,
    const float* __restrict__ bias, int64_t M, int K, int n_tiles, int num_tiles, int accumulate,
    const float* __restrict__ rowbias, int64_t ld_rowbias, const int64_t* __restrict__ seg,
    const float* __restrict__ a_amax, const float* __restrict__ b_scale_inv, const float* __restrict__ alpha,
    float* __restrict__ amax_out, float* __restrict__ stats_part) {
  constexpr int kPStages = kF16 ? kHStages : tc::kPStages;
  constexpr uint32_t P_STAGE_BYTES = kF16 ? H_STAGE_BYTES : tc::P_STAGE_BYTES;
  constexpr uint32_t A_BYTES = kF16 ? 2 * A_RAW_BYTES : A_RAW_BYTES;
  constexpr int BK = kF16 ? BKH : tc::BK;
  constexpr int kConvWarps = kF16 ? kHConvWarps : tc::kConvWarps;
  extern __shared__ uint8_t smem_dyn[];
  const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  const uint32_t out_stage = base + kPStages * P_STAGE_BYTES;       // 1024 B aligned (stages are 32 / 48 KB)
  const uint32_t bars = out_stage + kConvWarps * P_OUT_BYTES;
  // barriers (8 B each): full[6] | smem_empty[6] | a_ready[2] | a_empty[2] | acc_full | tmem ptr
  auto full = [&](int s) { return bars + 8u * s; };
  auto smem_empty = [&](int s) { return bars + 48u + 8u * s; };
  auto a_ready = [&](int t) { return bars + 96u + 8u * t; };
  auto a_empty = [&](int t) { return bars + 112u + 8u * t; };
  const uint32_t acc_full = bars + 128u;
  const uint32_t tmem_slot = bars + 136u;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = blockIdx.x;                            // rank in the pair = which 128 rows / which weight half
  const int num_kb = K / BK;
  // PERSISTENT: the pair walks tiles pair_id, pair_id + #pairs, ...; tile -> (row pair, N tile) with the N tiles of
  // one row pair adjacent, so that neighbouring pairs read the same A rows at the same time (L2 hit).  One launch
  // pays the prologue (barrier init, TMEM allocation, first TMA round trip: ~5k clk) once instead of once per tile
  // (measured 12k clk of fixed cost per 128 x 128 tile, more than the whole K = 256 mainloop); the TMA producer and
  // the MMA issuer run ahead into the next tile while the converter warps write the previous tile out.
  // Every role counts K blocks globally (`it`), which carries the barrier phases across tiles.

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b_hi));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b_lo));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_c));
    for (int s = 0; s < kPStages; ++s) {
      mbar_init(full(s), 1);
      mbar_init(smem_empty(s), 1 + kConvWarps);    // one multicast tcgen05.commit + one arrive per local converter warp
    }
    for (int t = 0; t < kPAStages; ++t) {
      mbar_init(a_ready(t), 2 * kConvWarps);       // converter warps of both CTAs (only the leader's copy is used)
      mbar_init(a_empty(t), 1);
    }
    mbar_init(acc_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tc_fence_before();
  cluster_sync_all();                                     // barriers of BOTH CTAs initialised, TMEM allocated
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (each CTA: its rows, its weight halves)
    if (lane == 0) {
      uint32_t it = 0;
      for (int tile = blockIdx.y; tile < num_tiles; tile += gridDim.y) {
        const int n0 = (tile % n_tiles) * BN;
        const int m0 = ((tile / n_tiles) * 2 + rank) * BM;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % kPStages;
          mbar_wait(smem_empty(s), ((it / kPStages) & 1) ^ 1);
          const uint32_t a_raw = base + s * P_STAGE_BYTES;
          mbar_arrive_expect_tx(full(s), P_STAGE_BYTES);
          tma_load_2d(a_raw, &map_a, kb * BK, m0, full(s));
          if (kF16) tma_load_2d(a_raw + A_RAW_BYTES, &map_a, kb * BK + 32, m0, full(s));
          tma_load_2d(a_raw + A_BYTES, &map_b_hi, kb * BK, n0 + 64 * rank, full(s));
          tma_load_2d(a_raw + A_BYTES + P_B_BYTES, &map_b_lo, kb * BK, n0 + 64 * rank, full(s));
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA only)
    // The whole warp walks the loop converged and ONE elected lane issues: under a divergent `if (lane == 0)` ptxas
    // wraps every tcgen05.mma in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop (~75 clk per MMA, measured 610 clk per K
    // block for the eight MMAs - as long as they take to execute).
    if (rank == 0) {
      const uint32_t leader = elect_one();
      uint32_t it = 0;
      for (int tile = blockIdx.y; tile < num_tiles; tile += gridDim.y) {
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % kPStages, t = it % kPAStages;
          mbar_wait(full(s), (it / kPStages) & 1);               // this CTA's tiles landed
          // both CTAs: tiles landed (their converters saw them) and A is in TMEM; for kb == 0 also: the converter
          // warps have finished reading the previous tile's accumulators (they run its epilogue first)
          mbar_wait(a_ready(t), (it / kPAStages) & 1);
          tc_fence_after();
          if (leader) {
            const uint64_t d_b = make_kmajor_sw128_desc(base + s * P_STAGE_BYTES + A_BYTES);
            const uint32_t a_hi = tmem_base + P_A_COL + t * 64;
            // four instructions per operand either way: K = 8 tf32 or K = 16 fp16 elements = 32 B of a weight row
            // and 8 tensor-memory columns of A per step
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t koff = static_cast<uint64_t>((k * 32) >> 4);
              const uint32_t acc = (kb > 0 || k > 0) ? 1u : 0u;
              if (kF16) {
                mma_f16_ts_pair(tmem_base + P_ACC1, a_hi + k * 8, d_b + koff, kPairDesc256H, acc);
                mma_f16_ts_pair(tmem_base + P_ACC2, a_hi + 32 + k * 8, d_b + koff, kPairDesc128H, acc);
              } else {
                mma_tf32_ts_pair(tmem_base + P_ACC1, a_hi + k * 8, d_b + koff, kPairDesc256, acc);        // A_hi . [B_hi ; B_lo]
                mma_tf32_ts_pair(tmem_base + P_ACC2, a_hi + 32 + k * 8, d_b + koff, kPairDesc128, acc);   // A_lo . B_hi
              }
            }
            tc_commit_pair(smem_empty(s));
            tc_commit_pair(a_empty(t));
            if (kb == num_kb - 1) tc_commit_pair(acc_full);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ------------------------------------------------------------ converters, then epilogue, per tile
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    uint32_t it = 0, tile_iter = 0;
    float a_scale = 1.f, out_scale = 1.f, out_max = 0.f;
    if (kF16) {
      a_scale = f16_scale(__ldg(a_amax));
      out_scale = (1.f / a_scale) * __ldg(b_scale_inv);       // powers of two: exact
    }
    for (int tile = blockIdx.y; tile < num_tiles; tile += gridDim.y, ++tile_iter) {
      const int n0 = (tile % n_tiles) * BN;
      const int64_t m0 = (static_cast<int64_t>(tile / n_tiles) * 2 + rank) * BM;
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const int s = it % kPStages, t = it % kPAStages;
        mbar_wait(full(s), (it / kPStages) & 1);
        uint32_t hi[16], lo[16];
        if (kF16) {
          // `half` = 0..3 here: 16 of the 64 K elements = four 16 B chunks of raw box half >> 1 -> 8 + 8 packed pairs
          const uint32_t row_addr = base + s * P_STAGE_BYTES + (half >> 1) * A_RAW_BYTES + r * 128;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float4 v;
            const uint32_t addr = row_addr + (((4 * (half & 1) + c) ^ (r & 7)) << 4);    // undo the 128 B TMA swizzle
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
            split_f16x2(v.x * a_scale, v.y * a_scale, hi[2 * c], lo[2 * c]);
            split_f16x2(v.z * a_scale, v.w * a_scale, hi[2 * c + 1], lo[2 * c + 1]);
          }
        } else {
          const uint32_t row_addr = base + s * P_STAGE_BYTES + r * 128;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float4 v;
            const uint32_t addr = row_addr + (((4 * half + c) ^ (r & 7)) << 4);          // undo the 128 B TMA swizzle
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
            const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) split_tf32(e[i], hi[4 * c + i], lo[4 * c + i]);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_empty(s));
        mbar_wait(a_empty(t), ((it / kPAStages) & 1) ^ 1);
        tc_fence_after();
        if (kF16) {
          const uint32_t a_hi = tmem_base + lane_addr + P_A_COL + t * 64 + 8 * half;
          const uint32_t (&h8)[8] = *reinterpret_cast<const uint32_t(*)[8]>(hi);
          const uint32_t (&l8)[8] = *reinterpret_cast<const uint32_t(*)[8]>(lo);
          tmem_st8(a_hi, h8);
          tmem_st8(a_hi + 32, l8);
        } else {
          const uint32_t a_hi = tmem_base + lane_addr + P_A_COL + t * 64 + 16 * half;
          tmem_st16(a_hi, hi);
          tmem_st16(a_hi + 32, lo);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(a_ready(t));
      }
      mbar_wait(acc_full, tile_iter & 1);
      tc_fence_after();
      const int64_t row = m0 + r;
      const float* rb = (rowbias && row < M) ? rowbias + __ldg(seg + row) * ld_rowbias + n0 : nullptr;
      // Each warp writes its 32 x 32 boxes through shared memory and a TMA store (a reduce-add store when the
      // result accumulates into C): row-per-thread global stores touch 32 lines per instruction (4096 LSU wavefronts
      // per tile; ncu: the tensor pipe idled ~7 k clk per tile behind them), the staged box is eight conflict-free
      // 128-bit shared stores per thread and one bulk copy that drains while the warp is already converting the
      // next tile.  Rows past M are clipped by the tensor map.
      const uint32_t sbuf = out_stage + (warp - 2) * P_OUT_BYTES;
      if (kF16) {
        // one 32 x 32 box per warp (columns [32 * half, +32)), read from tensor memory in two halves of 16 columns
        const int c0 = half * 32;
        const uint32_t mcol = c0 < 64 ? c0 : 64 + c0;
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the previous box has left this buffer
        __syncwarp();
#pragma unroll 1
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t v[16], w[16], u[16];
          tmem_ld16(tmem_base + lane_addr + P_ACC1 + mcol + 16 * hh, v);
          tmem_ld16(tmem_base + lane_addr + P_ACC1 + mcol + 64 + 16 * hh, w);
          tmem_ld16(tmem_base + lane_addr + P_ACC2 + c0 + 16 * hh, u);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            // the correction accumulators carry the 2^11 of the low parts; then undo the operand scales
            float4 o = make_float4(fmaf(__uint_as_float(w[4 * q]) + __uint_as_float(u[4 * q]), 1.f / 2048.f, __uint_as_float(v[4 * q])) * out_scale,
                                   fmaf(__uint_as_float(w[4 * q + 1]) + __uint_as_float(u[4 * q + 1]), 1.f / 2048.f, __uint_as_float(v[4 * q + 1])) * out_scale,
                                   fmaf(__uint_as_float(w[4 * q + 2]) + __uint_as_float(u[4 * q + 2]), 1.f / 2048.f, __uint_as_float(v[4 * q + 2])) * out_scale,
                                   fmaf(__uint_as_float(w[4 * q + 3]) + __uint_as_float(u[4 * q + 3]), 1.f / 2048.f, __uint_as_float(v[4 * q + 3])) * out_scale);
            const int qq = 4 * hh + q;
            if (bias) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(bias + n0 + c0) + qq);
              o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
            }
            if (rb) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(rb + c0) + qq);
              o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
            }
            if (alpha) {                                     // inference: BatchNorm is folded into W / bias, PReLU here
              const float4 al = __ldg(reinterpret_cast<const float4*>(alpha + n0 + c0) + qq);
              o.x = o.x > 0.f ? o.x : al.x * o.x; o.y = o.y > 0.f ? o.y : al.y * o.y;
              o.z = o.z > 0.f ? o.z : al.z * o.z; o.w = o.w > 0.f ? o.w : al.w * o.w;
            }
            if (amax_out && row < M) out_max = amax4(out_max, o);
            const uint32_t dst = sbuf + lane * 128 + ((qq ^ (lane & 7)) << 4);          // SWIZZLE_128B box layout
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w) : "memory");
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          const int crow = static_cast<int>(m0) + quarter * 32;
          if (crow < M) {
            if (accumulate) tma_reduce_add_2d(&map_c, sbuf, n0 + c0, crow);
            else tma_store_2d(&map_c, sbuf, n0 + c0, crow);
          }
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        // BatchNorm statistics of the layer's output without another pass over it: lane c reduces column c of the staged
        // box (its 32 rows; rows past M excluded) to {group mean, sum of squared deviations from it}.  The sums are taken
        // relative to the column's first row of the group (a pivot within one standard deviation or so of the values), so
        // no large squares are subtracted from each other anywhere: Keras' two-pass variance is reproduced to fp32
        // rounding also when |mean| >> std.  bn_stats_from_partials combines the groups in fp64 (mean_g, M2_g, n_g).
        // The swizzled box is read conflict-free (one 128 B row per step).
        const int64_t grow = m0 + quarter * 32;
        if (stats_part && grow < M) {
          float ssum = 0.f, ssq = 0.f, pivot = 0.f;
#pragma unroll 8
          for (int rr = 0; rr < 32; ++rr) {
            float hv;
            const uint32_t src = sbuf + rr * 128 + ((((lane >> 2) ^ (rr & 7))) << 4) + (lane & 3) * 4;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(hv) : "r"(src));
            if (rr == 0) pivot = hv;
            if (grow + rr < M) {
              const float d = hv - pivot;
              ssum += d;
              ssq = fmaf(d, d, ssq);
            }
          }
          const float cnt = static_cast<float>(M - grow < 32 ? M - grow : 32);
          const float dm = ssum / cnt;
          reinterpret_cast<float2*>(stats_part)[(grow >> 5) * (static_cast<int64_t>(n_tiles) * BN) + n0 + c0 + lane] =
              make_float2(pivot + dm, fmaxf(ssq - ssum * dm, 0.f));
        }
      } else {
  #pragma unroll 1
        for (int c0 = half * (BN / 2); c0 < (half + 1) * (BN / 2); c0 += 32) {
          uint32_t v[32], w[32], u[32];
          const uint32_t mcol = c0 < 64 ? c0 : 64 + c0;        // [0,64) -> [0,64), [64,128) -> [128,192)
          tmem_ld32(tmem_base + lane_addr + P_ACC1 + mcol, v);
          tmem_ld32(tmem_base + lane_addr + P_ACC1 + mcol + 64, w);
          tmem_ld32(tmem_base + lane_addr + P_ACC2 + c0, u);
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the previous box has left this buffer
          __syncwarp();
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  #pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 o = make_float4(__uint_as_float(v[4 * q]) + (__uint_as_float(w[4 * q]) + __uint_as_float(u[4 * q])),
                                   __uint_as_float(v[4 * q + 1]) + (__uint_as_float(w[4 * q + 1]) + __uint_as_float(u[4 * q + 1])),
                                   __uint_as_float(v[4 * q + 2]) + (__uint_as_float(w[4 * q + 2]) + __uint_as_float(u[4 * q + 2])),
                                   __uint_as_float(v[4 * q + 3]) + (__uint_as_float(w[4 * q + 3]) + __uint_as_float(u[4 * q + 3])));
            if (bias) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(bias + n0 + c0) + q);
              o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
            }
            if (rb) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(rb + c0) + q);
              o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
            }
            const uint32_t dst = sbuf + lane * 128 + ((q ^ (lane & 7)) << 4);          // SWIZZLE_128B box layout
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "f"(o.x), "f"(o.y), "f"(o.z), "f"(o.w) : "memory");
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            const int crow = static_cast<int>(m0) + quarter * 32;
            if (crow < M) {
              if (accumulate) tma_reduce_add_2d(&map_c, sbuf, n0 + c0, crow);
              else tma_store_2d(&map_c, sbuf, n0 + c0, crow);
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      }
      tc_fence_before();          // accumulator reads ordered before this warp's next a_ready arrive
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");           // every box written before the CTA exits
    if (kF16) amax_commit(out_max, amax_out);
  }
  tc_fence_before();
  cluster_sync_all();              // the peer's tensor core may still read this CTA's shared memory until its commits land
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
  }
}

// ---------------------------------------------------------------------------------------------
// fp16 forward / dX kernel for widths that are multiples of 256: one CTA pair computes a 256 x 256 tile per pass.
//
// linear_tc_pair_kernel<true> computes 256 x 128 tiles, so a 256-wide output fetches every raw fp32 A row from L2 twice
// and splits it twice: per CTA and K block of 64, 2 x (32 KB raw A + 16 KB weight halves) = 96 KB of L2 -> SM ingest,
// the bound of that kernel.  Here both 128-column halves come out of one pass over A: 32 KB raw A + 32 KB weight halves
// = 64 KB per K block, for the same tensor work.  Tensor memory then holds nothing but the two accumulators, so the
// split A operand lives in shared memory (SS-form MMAs):
//   TMEM (each CTA, its 128 rows):  MAIN = A_hi.B_hi in columns [0, 256), CORR = A_hi.B_lo + A_lo.B_hi in [256, 512)
//   (both correction products carry the same 2^11, so one accumulator takes both; the epilogue adds CORR * 2^-11).
//   Per CTA and stage: [A raw box k0..k0+31 | A raw box k0+32..k0+63 | B_hi 128 x 64 | B_lo 128 x 64]  = 64 KB
//   (rank r holds output columns [128 r, 128 r + 128) of the pass: cta_group::2 takes N = 256 as two halves).
// The converters split A IN PLACE: A_hi over raw box 0 and A_lo over raw box 1, each a K-major SWIZZLE_128B fp16
// operand of 128 rows x 128 B (the layout TMA gives the weight tiles).  Row r of both the raw boxes and the split
// operands is the 128 B at r * 128, and only the four converter warps of r's lane quarter touch it: they meet at a
// named barrier between reading their raw chunks and writing the split ones.  The stage is released by the MMA commit.
// Three 64 KB stages + 16 x 2 KB of epilogue staging fit the 227 KB; there is no room for a second accumulator set,
// so (as in linear_tc_pair_kernel) the converters write a tile out before they feed the next one.
constexpr int kSStages = 3;
constexpr uint32_t S_B_BYTES = 128 * BKH * 2;                         // 16 KB: 128 weight rows of one half
constexpr uint32_t S_STAGE_BYTES = 2 * A_RAW_BYTES + 2 * S_B_BYTES;   // 64 KB
constexpr uint32_t S_OUT_BYTES = 32 * 16 * 4;                         // per converter warp: one 32 x 16 output box
constexpr uint32_t kSSmemBytes = kSStages * S_STAGE_BYTES + kHConvWarps * S_OUT_BYTES + 1024 + 256;
static_assert(kSSmemBytes <= 232448, "fp16 256-column kernel exceeds the 227 KB of shared memory per CTA");
constexpr uint32_t S_MAIN = 0, S_CORR = 256;

__device__ __forceinline__ void mma_f16_ss_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kHThreads, 1) linear_f16_pass256_kernel(
    const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b_hi,
    const __grid_constant__ CUtensorMap map_b_lo, const __grid_constant__ CUtensorMap map_c,
    const float* __restrict__ bias, int64_t M, int K, int N, int num_tiles, int accumulate,
    const float* __restrict__ rowbias, int64_t ld_rowbias, const int64_t* __restrict__ seg,
    const float* __restrict__ a_amax, const float* __restrict__ b_scale_inv, const float* __restrict__ alpha,
    float* __restrict__ amax_out, float* __restrict__ stats_part) {
  extern __shared__ uint8_t smem_dyn[];
  const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  const uint32_t out_stage = base + kSStages * S_STAGE_BYTES;     // 1024 B aligned
  const uint32_t bars = out_stage + kHConvWarps * S_OUT_BYTES;
  // barriers (8 B each): full[3] | smem_empty[3] | a_ready[3] | acc_full | tmem ptr
  auto full = [&](int s) { return bars + 8u * s; };
  auto smem_empty = [&](int s) { return bars + 24u + 8u * s; };
  auto a_ready = [&](int s) { return bars + 48u + 8u * s; };
  const uint32_t acc_full = bars + 72u;
  const uint32_t tmem_slot = bars + 80u;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = blockIdx.x;
  const int num_kb = K / BKH;
  const int n_pass = N / 256;
  // persistent walk as in linear_tc_pair_kernel: tile -> (row pair, 256-column pass), the passes of a row pair adjacent

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b_hi));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b_lo));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_c));
    for (int s = 0; s < kSStages; ++s) {
      mbar_init(full(s), 1);
      mbar_init(smem_empty(s), 1);                 // the multicast tcgen05.commit: the split A is read by the MMAs alone
      mbar_init(a_ready(s), 2 * kHConvWarps);      // converter warps of both CTAs (only the leader's copy is used)
    }
    mbar_init(acc_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      uint32_t it = 0;
      for (int tile = blockIdx.y; tile < num_tiles; tile += gridDim.y) {
        const int n0 = (tile % n_pass) * 256;
        const int m0 = ((tile / n_pass) * 2 + rank) * BM;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % kSStages;
          mbar_wait(smem_empty(s), ((it / kSStages) & 1) ^ 1);
          const uint32_t st = base + s * S_STAGE_BYTES;
          mbar_arrive_expect_tx(full(s), S_STAGE_BYTES);
          tma_load_2d(st, &map_a, kb * BKH, m0, full(s));
          tma_load_2d(st + A_RAW_BYTES, &map_a, kb * BKH + 32, m0, full(s));
          tma_load_2d(st + 2 * A_RAW_BYTES, &map_b_hi, kb * BKH, n0 + 128 * rank, full(s));
          tma_load_2d(st + 2 * A_RAW_BYTES + S_B_BYTES, &map_b_lo, kb * BKH, n0 + 128 * rank, full(s));
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA only; converged warp, one elected lane)
    if (rank == 0) {
      const uint32_t leader = elect_one();
      uint32_t it = 0;
      for (int tile = blockIdx.y; tile < num_tiles; tile += gridDim.y) {
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const int s = it % kSStages;
          const uint32_t ph = (it / kSStages) & 1;
          mbar_wait(full(s), ph);
          // both CTAs: stage landed and split; for kb == 0 also: the previous tile's accumulators have been read
          mbar_wait(a_ready(s), ph);
          tc_fence_after();
          if (leader) {
            const uint32_t st = base + s * S_STAGE_BYTES;
            const uint64_t d_ahi = make_kmajor_sw128_desc(st);
            const uint64_t d_alo = make_kmajor_sw128_desc(st + A_RAW_BYTES);
            const uint64_t d_bhi = make_kmajor_sw128_desc(st + 2 * A_RAW_BYTES);
            const uint64_t d_blo = make_kmajor_sw128_desc(st + 2 * A_RAW_BYTES + S_B_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k) {               // K = 16 per instruction: 32 B of each 128 B operand row
              const uint64_t koff = static_cast<uint64_t>((k * 32) >> 4);
              const uint32_t acc = (kb > 0 || k > 0) ? 1u : 0u;
              mma_f16_ss_pair(tmem_base + S_MAIN, d_ahi + koff, d_bhi + koff, kPairDesc256H, acc);
              mma_f16_ss_pair(tmem_base + S_CORR, d_ahi + koff, d_blo + koff, kPairDesc256H, acc);
              mma_f16_ss_pair(tmem_base + S_CORR, d_alo + koff, d_bhi + koff, kPairDesc256H, 1u);
            }
            tc_commit_pair(smem_empty(s));
            if (kb == num_kb - 1) tc_commit_pair(acc_full);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ------------------------------------------------------------ converters, then epilogue, per tile
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;                  // 0..3: which 16 of the 64 K elements; which 64 output columns
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    uint32_t it = 0, tile_iter = 0;
    const float a_scale = f16_scale(__ldg(a_amax));
    const float out_scale = (1.f / a_scale) * __ldg(b_scale_inv);     // powers of two: exact
    float out_max = 0.f;
    for (int tile = blockIdx.y; tile < num_tiles; tile += gridDim.y, ++tile_iter) {
      const int n0 = (tile % n_pass) * 256;
      const int64_t m0 = (static_cast<int64_t>(tile / n_pass) * 2 + rank) * BM;
      for (int kb = 0; kb < num_kb; ++kb, ++it) {
        const int s = it % kSStages;
        mbar_wait(full(s), (it / kSStages) & 1);
        const uint32_t st = base + s * S_STAGE_BYTES;
        uint32_t hi[8], lo[8];
        // the row's swizzled addresses are recomputed per K block (a few integer instructions): hoisted out of the
        // tile loops, ptxas kept them in local memory
        uint32_t rr7;
        asm volatile("and.b32 %0, %1, 7;" : "=r"(rr7) : "r"(r));
        const uint32_t raw_row = st + (half >> 1) * A_RAW_BYTES + r * 128;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float4 v;
          const uint32_t addr = raw_row + (((4 * (half & 1) + c) ^ rr7) << 4);          // undo the 128 B TMA swizzle
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
          split_f16x2(v.x * a_scale, v.y * a_scale, hi[2 * c], lo[2 * c]);
          split_f16x2(v.z * a_scale, v.w * a_scale, hi[2 * c + 1], lo[2 * c + 1]);
        }
        // the four warps of this lane quarter have read rows r of both raw boxes before any of them overwrites them
        asm volatile("bar.sync %0, 128;" ::"r"(1 + quarter) : "memory");
        // K elements 16 * half .. + 15 are the 16 B chunks 2 * half, 2 * half + 1 of the fp16 row (SWIZZLE_128B)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const uint32_t off = r * 128 + (((2 * half + j) ^ rr7) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};"
                       ::"r"(st + off), "r"(hi[4 * j]), "r"(hi[4 * j + 1]), "r"(hi[4 * j + 2]), "r"(hi[4 * j + 3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};"
                       ::"r"(st + A_RAW_BYTES + off), "r"(lo[4 * j]), "r"(lo[4 * j + 1]), "r"(lo[4 * j + 2]), "r"(lo[4 * j + 3]) : "memory");
        }
        // Hand-off of the split operand to the tensor core.  Each SM of the pair reads the A rows of its OWN CTA's shared
        // memory (cta_group::2 splits M = 256 into the two CTAs' 128 rows), so every converter orders its generic-proxy
        // stores before async-proxy reads of its own CTA's shared memory with fence.proxy.async.shared::cta, and only the
        // signal crosses the pair: the arrive below (a default, i.e. .release.cta, remote arrive, as for the tensor-memory
        // A of linear_tc_pair_kernel) is program-ordered after the fence, the leader issues the MMAs only after the phase
        // completed, and the MMA's reads of this CTA's rows are performed by this SM's tensor core, through the proxy the
        // fence has already made the stores visible to.  No generic-proxy data crosses the CTA boundary, so no
        // cluster-scope release is needed (it costs a MEMBAR.ALL.GPU per arrive: see mbar_arrive_leader).
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(a_ready(s));
      }
      mbar_wait(acc_full, tile_iter & 1);
      tc_fence_after();
      const int64_t row = m0 + r;
      const float* rb = (rowbias && row < M) ? rowbias + __ldg(seg + row) * ld_rowbias + n0 : nullptr;
      const int crow = static_cast<int>(m0) + quarter * 32;
      const int64_t grow = m0 + quarter * 32;
      // 64 output columns per warp as four 32 x 16 boxes through a 2 KB staging buffer and TMA stores (SWIZZLE_64B: the
      // 16 B chunk index XOR bits 1-2 of the row, so the row-per-lane stores are conflict-free)
      const uint32_t sbuf = out_stage + (warp - 2) * S_OUT_BYTES;
#pragma unroll 1
      for (int b = 0; b < 4; ++b) {
        const int c0 = half * 64 + b * 16;
        uint32_t v[16], w[16];
        tmem_ld16(tmem_base + lane_addr + S_MAIN + c0, v);
        tmem_ld16(tmem_base + lane_addr + S_CORR + c0, w);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        float4 o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          // the correction accumulator carries the 2^11 of the low parts; then undo the operand scales
          o[q] = make_float4(fmaf(__uint_as_float(w[4 * q]), 1.f / 2048.f, __uint_as_float(v[4 * q])) * out_scale,
                             fmaf(__uint_as_float(w[4 * q + 1]), 1.f / 2048.f, __uint_as_float(v[4 * q + 1])) * out_scale,
                             fmaf(__uint_as_float(w[4 * q + 2]), 1.f / 2048.f, __uint_as_float(v[4 * q + 2])) * out_scale,
                             fmaf(__uint_as_float(w[4 * q + 3]), 1.f / 2048.f, __uint_as_float(v[4 * q + 3])) * out_scale);
          if (bias) {
            const float4 bb = __ldg(reinterpret_cast<const float4*>(bias + n0 + c0) + q);
            o[q].x += bb.x; o[q].y += bb.y; o[q].z += bb.z; o[q].w += bb.w;
          }
          if (rb) {
            const float4 bb = __ldg(reinterpret_cast<const float4*>(rb + c0) + q);
            o[q].x += bb.x; o[q].y += bb.y; o[q].z += bb.z; o[q].w += bb.w;
          }
          if (alpha) {                                       // inference: BatchNorm is folded into W / bias, PReLU here
            const float4 al = __ldg(reinterpret_cast<const float4*>(alpha + n0 + c0) + q);
            o[q].x = o[q].x > 0.f ? o[q].x : al.x * o[q].x; o[q].y = o[q].y > 0.f ? o[q].y : al.y * o[q].y;
            o[q].z = o[q].z > 0.f ? o[q].z : al.z * o[q].z; o[q].w = o[q].w > 0.f ? o[q].w : al.w * o[q].w;
          }
          if (amax_out && row < M) out_max = amax4(out_max, o[q]);
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the previous box has left the buffer
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t dst = sbuf + lane * 64 + ((q ^ ((lane >> 1) & 3)) << 4);      // SWIZZLE_64B box layout
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "f"(o[q].x), "f"(o[q].y), "f"(o[q].z), "f"(o[q].w) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          if (crow < M) {
            if (accumulate) tma_reduce_add_2d(&map_c, sbuf, n0 + c0, crow);
            else tma_store_2d(&map_c, sbuf, n0 + c0, crow);
          }
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        // BatchNorm statistics of the box's 32-row group, pivot-shifted as in linear_tc_pair_kernel: lane c < 16 reduces
        // column c (the same order of sums as there)
        if (stats_part && grow < M && lane < 16) {
          float ssum = 0.f, ssq = 0.f, pivot = 0.f;
#pragma unroll 8
          for (int rr = 0; rr < 32; ++rr) {
            float hv;
            const uint32_t src = sbuf + rr * 64 + (((lane >> 2) ^ ((rr >> 1) & 3)) << 4) + (lane & 3) * 4;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(hv) : "r"(src));
            if (rr == 0) pivot = hv;
            if (grow + rr < M) {
              const float d = hv - pivot;
              ssum += d;
              ssq = fmaf(d, d, ssq);
            }
          }
          const float cnt = static_cast<float>(M - grow < 32 ? M - grow : 32);
          const float dm = ssum / cnt;
          reinterpret_cast<float2*>(stats_part)[(grow >> 5) * static_cast<int64_t>(N) + n0 + c0 + lane] =
              make_float2(pivot + dm, fmaxf(ssq - ssum * dm, 0.f));
        }
        __syncwarp();
      }
      tc_fence_before();          // accumulator reads ordered before this warp's next a_ready arrive
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");           // every box written before the CTA exits
    amax_commit(out_max, amax_out);
  }
  tc_fence_before();
  cluster_sync_all();              // the peer's tensor core may still read this CTA's shared memory until its commits land
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
  }
}

// hi = rna_tf32(w), lo = rna_tf32(w - hi); optionally transposed so that the reduction index
// is contiguous (the K-major layout the B operand wants).
// W is a [rows, cols] block with row pitch ldw; element (r, c) goes to out[r*ldo + c] or, transposed,
// to out[c*ldo + r].
__global__ void __launch_bounds__(256) split_weights_kernel(const float* __restrict__ W, int rows, int cols, int64_t ldw,
                                                            int transpose, int64_t ldo, float* __restrict__ hi,
                                                            float* __restrict__ lo) {
  const int64_t n = static_cast<int64_t>(rows) * cols;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i - static_cast<int64_t>(r) * cols);
    const float w = __ldg(W + r * ldw + c);
    const float h = __uint_as_float(rna_tf32(w));
    const float l = __uint_as_float(rna_tf32(w - h));
    const int64_t o = transpose ? c * ldo + r : r * ldo + c;
    hi[o] = h;
    lo[o] = l;
  }
}

// |max| of a strided matrix into *cell (pre-zeroed; non-negative floats order like their bit patterns).
__device__ __forceinline__ void absmax_body(const float* __restrict__ A, int64_t lda, int64_t M, int K, float* cell,
                                            const float* __restrict__ col_scale) {
  float m = 0.f;
  for (int64_t r = blockIdx.x; r < M; r += gridDim.x) {
    const float* row = A + r * lda;
    for (int c = threadIdx.x; c < K; c += blockDim.x)
      m = fmaxf(m, fabsf(col_scale ? __ldg(row + c) * __ldg(col_scale + c) : __ldg(row + c)));
  }
  amax_commit(m, cell);
}
__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ A, int64_t lda, int64_t M, int K, float* cell,
                                                     const float* __restrict__ col_scale) {
  absmax_body(A, lda, M, K, cell, col_scale);
}

// Inference fold of BatchNorm into the bias of the dense layer in front of it: b' = b * scale + shift.
__global__ void fold_bias_kernel(const float* __restrict__ bias, const float* __restrict__ scale, const float* __restrict__ shift,
                                 int N, float* __restrict__ out) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n < N) out[n] = fmaf(bias ? bias[n] : 0.f, scale[n], shift[n]);
}

// cell = max(cell, other): joins the |max| a fused GEMM produced into the running maximum it read its own scale from.
__global__ void amax_merge_kernel(float* cell, const float* other) {
  if (*other > *cell) *cell = *other;
}

// fp16 split of the weights for linear_tc_pair_kernel<true>: hi = fp16(w * s), lo = fp16((w * s - hi) * 2^11) with
// s = f16_scale(*amax); *scale_inv = 1 / s for the epilogue.
__device__ __forceinline__ void split_weights_f16_body(const float* __restrict__ W, int rows, int cols, int64_t ldw,
                                                       int transpose, int64_t ldo, __half* __restrict__ hi,
                                                       __half* __restrict__ lo, const float* __restrict__ amax,
                                                       float* __restrict__ scale_inv, const float* __restrict__ col_scale) {
  const float s = f16_scale(__ldg(amax));
  if (blockIdx.x == 0 && threadIdx.x == 0) *scale_inv = 1.f / s;
  const int64_t n = static_cast<int64_t>(rows) * cols;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i - static_cast<int64_t>(r) * cols);
    const float w = col_scale ? __ldg(W + r * ldw + c) * __ldg(col_scale + c) : __ldg(W + r * ldw + c);
    const float y = w * s;
    const __half h = __float2half_rn(y);
    const int64_t o = transpose ? c * ldo + r : r * ldo + c;
    hi[o] = h;
    lo[o] = __float2half_rn((y - __half2float(h)) * 2048.f);
  }
}
__global__ void __launch_bounds__(256) split_weights_f16_kernel(const float* __restrict__ W, int rows, int cols, int64_t ldw,
                                                                int transpose, int64_t ldo, __half* __restrict__ hi,
                                                                __half* __restrict__ lo, const float* __restrict__ amax,
                                                                float* __restrict__ scale_inv,
                                                                const float* __restrict__ col_scale) {
  split_weights_f16_body(W, rows, cols, ldw, transpose, ldo, hi, lo, amax, scale_inv, col_scale);
}

// All weight blocks of a train step in two launches (blockIdx.y = job): the |max| cells first (several blocks may share
// one cell: the blocks of a concatenated operand), then the splits.  The per-GEMM form above costs a memset, a |max|
// kernel and a split kernel per weight block - ~45 launches of a few microseconds each per step at the default
// architecture, every one of them a bubble between two large kernels.
__global__ void __launch_bounds__(256) absmax_multi_kernel(const __grid_constant__ SplitJobs jobs) {
  const SplitJob& j = jobs.j[blockIdx.y];
  absmax_body(j.W, j.ldw, j.rows, j.cols, j.cells, nullptr);
}
__global__ void __launch_bounds__(256) split_weights_f16_multi_kernel(const __grid_constant__ SplitJobs jobs) {
  const SplitJob& j = jobs.j[blockIdx.y];
  split_weights_f16_body(j.W, j.rows, j.cols, j.ldw, j.transpose, j.ldo, static_cast<__half*>(j.hi), static_cast<__half*>(j.lo),
                         j.cells, j.cells + 1, nullptr);
}

// ---------------------------------------------------------------------------------------------
// Weight gradient  dW[K_in, N] = A[M, K_in]^T . dH[M, N]  on the tensor cores.
//
// The reduction runs over the M rows, both operands are activations (split on the fly) and both
// are stored with the reduction index as the SLOW dimension.  One CTA = one 128 x 128 tile of dW
// over a range of rows, 448 threads:
//   warp 0      TMA: per 32-row step the raw A slab [32 x 128] (no swizzle) and the raw dH slab as
//               four [32 x 32] boxes (SWIZZLE_128B_ATOM_32B = the canonical MN-major fp32 layout)
//   warp 1      MMA issuer: A^T from tensor memory (K-major by construction), dH from shared
//               memory as an MN-major operand; 2 MMAs per K=8 step (N = 256 into [main | correction],
//               N = 128 into correction); owns TMEM
//   warps 2-5   A^T converters: thread i gathers column i of the A slab (32 conflict-free scalar
//               loads: the transpose is free), splits it and writes both halves into TMEM
//   warps 6-9   dH splitters: the slab is split element-wise in place (hi) + the buffer right behind
//               it (lo), then fence.proxy.async hands both to the tensor core
//   warps 10-13 accumulators: every 16 steps (512 rows) they fold main + correction into a
//               running fp32 sum kept in TMEM columns [384, 512) with round-to-nearest adds, so
//               that no truncating tensor-core chain is longer than 128 K-steps; at the end they
//               write the CTA's partial tile.  Partials are summed in a fixed order afterwards.
static int g_wg_chain = 16;                              // K blocks (of 32 rows) per tensor-core accumulation chain
void set_wgrad_chain(int c) { if (c > 0) g_wg_chain = c; }
constexpr int kWgThreads = 448;
constexpr uint32_t WG_X_BYTES = 32 * 128 * 4;            // 16 KB raw A slab
constexpr uint32_t WG_Y_BYTES = 32 * 128 * 4;            // 16 KB dH slab (hi in place) ; + 16 KB lo
constexpr uint32_t WG_STAGE_BYTES = WG_X_BYTES + 2 * WG_Y_BYTES;
constexpr uint32_t kWgSmemBytes = kStages * WG_STAGE_BYTES + 1024 + 256;
constexpr uint32_t RUN_COL = 384;
// D = F32, A = B = TF32, A K-major (TMEM), B MN-major, N = 128, M = 128
constexpr uint32_t kWgInstrDesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | (static_cast<uint32_t>(128 >> 3) << 17) |
                                  (static_cast<uint32_t>(128 >> 4) << 24);
constexpr uint32_t kWgInstrDesc2N = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | (static_cast<uint32_t>(256 >> 3) << 17) |
                                    (static_cast<uint32_t>(128 >> 4) << 24);

// MN-major fp32 operand, SWIZZLE_128B_BASE32B: 128 B rows (32 elements along N), 4-row swizzle
// groups 512 B apart along K, 32-column boxes 4096 B apart along N.
__device__ __forceinline__ uint64_t make_mnmajor_b32_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>(4096 >> 4) << 16;                    // leading byte offset: next 32-column box
  d |= static_cast<uint64_t>(512 >> 4) << 32;                     // stride byte offset: next 4-row group
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(1) << 61;                            // SWIZZLE_128B_BASE32B
  return d;
}

__global__ void __launch_bounds__(kWgThreads, 1) wgrad_tc_kernel(
    const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_y,
    float* __restrict__ out, int64_t out_split_stride, int ldo, int num_kb_total, int kb_per_split, int kWgChain,
    int k_rows) {
  extern __shared__ uint8_t smem_dyn[];
  const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  const uint32_t bars = base + kStages * WG_STAGE_BYTES;
  auto full = [&](int s) { return bars + 8u * s; };
  auto smem_empty = [&](int s) { return bars + 32u + 8u * s; };
  auto a_ready = [&](int t) { return bars + 64u + 8u * t; };
  auto a_empty = [&](int t) { return bars + 80u + 8u * t; };
  const uint32_t acc_full = bars + 96u, acc_empty = bars + 104u, tmem_slot = bars + 112u;
  auto y_ready = [&](int s) { return bars + 120u + 8u * s; };      // dH slab of smem stage s is split

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i0 = blockIdx.x * 128, j0 = blockIdx.y * 128;
  const int kb_begin = blockIdx.z * kb_per_split;
  const int kb_end = min(num_kb_total, kb_begin + kb_per_split);
  const int num_kb = kb_end - kb_begin;                 // host guarantees >= 1
  out += static_cast<int64_t>(blockIdx.z) * out_split_stride;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_y));
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full(s), 1);
      mbar_init(smem_empty(s), 1);
      mbar_init(y_ready(s), 128);
    }
    for (int t = 0; t < kWgAStages; ++t) {
      mbar_init(a_ready(t), 128);
      mbar_init(a_empty(t), 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kStages;
        mbar_wait(smem_empty(s), ((kb / kStages) & 1) ^ 1);
        const uint32_t xs = base + s * WG_STAGE_BYTES;
        const int m = (kb_begin + kb) * 32;
        mbar_arrive_expect_tx(full(s), WG_X_BYTES + WG_Y_BYTES);
        tma_load_2d(xs, &map_x, i0, m, full(s));
#pragma unroll
        for (int b = 0; b < 4; ++b) tma_load_2d(xs + WG_X_BYTES + b * 4096, &map_y, j0 + 32 * b, m, full(s));
      }
    }
  } else if (warp == 1) {
    const uint32_t leader = elect_one();             // converged warp, one elected lane issues (see linear_tc_kernel)
    for (int kb = 0; kb < num_kb; ++kb) {
      const int s = kb % kStages, t = kb % kWgAStages;
      const int chain = kb / kWgChain, pos = kb % kWgChain;
      if (pos == 0 && chain > 0) mbar_wait(acc_empty, (chain - 1) & 1);   // accumulators drained
      mbar_wait(a_ready(t), (kb / kWgAStages) & 1);     // A^T of this step is in tensor memory
      mbar_wait(y_ready(s), (kb / kStages) & 1);        // dH slab of this step is split (hi in place, lo right behind it)
      tc_fence_after();
      if (leader) {
        const uint32_t y_hi = base + s * WG_STAGE_BYTES + WG_X_BYTES;
        const uint64_t d_hi = make_mnmajor_b32_desc(y_hi);
        const uint32_t a_hi = tmem_base + A_COL + t * 64;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint64_t koff = static_cast<uint64_t>((k * 8 * 128) >> 4);       // 8 rows of 128 B per K step
          const uint32_t acc = (pos > 0 || k > 0) ? 1u : 0u;
          // The lo slab lies right behind the hi slab, i.e. [dH_hi | dH_lo] is ONE MN-major operand of eight 32-column
          // boxes: A_hi meets both in a single N = 256 instruction whose accumulator is [main | correction]; A_lo . dH_hi
          // then adds into the correction half (in-order execution).  Eight instead of twelve issues per K block.
          mma_tf32_ts(tmem_base + ACC_MAIN, a_hi + k * 8, d_hi + koff, kWgInstrDesc2N, acc);
          mma_tf32_ts(tmem_base + ACC_CORR, a_hi + 32 + k * 8, d_hi + koff, kWgInstrDesc, 1u);
        }
        tc_commit(smem_empty(s));
        tc_commit(a_empty(t));
        if (pos == kWgChain - 1 || kb == num_kb - 1) tc_commit(acc_full);
      }
      __syncwarp();
    }
  } else if (warp < 6) {
    // ------------------------------------------------------------ A^T converters: column i of the A slab -> TMEM
    const int quarter = warp & 3;
    const int i = quarter * 32 + lane;                 // output row (column of the A slab) owned by this thread
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    for (int kb = 0; kb < num_kb; ++kb) {
      const int s = kb % kStages, t = kb % kWgAStages;
      mbar_wait(full(s), (kb / kStages) & 1);
      const uint32_t xs = base + s * WG_STAGE_BYTES;
      uint32_t hi[32], lo[32];
#pragma unroll
      for (int m = 0; m < 32; ++m) {
        float v;
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(xs + (m * 128 + i) * 4));
        split_tf32(v, hi[m], lo[m]);
      }
      mbar_wait(a_empty(t), ((kb / kWgAStages) & 1) ^ 1);
      tc_fence_after();
      const uint32_t a_hi = tmem_base + lane_addr + A_COL + t * 64;
      tmem_st32(a_hi, hi);
      tmem_st32(a_hi + 32, lo);
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      mbar_arrive(a_ready(t));
    }
  } else if (warp < 10) {
    // ------------------------------------------------------------ dH splitters: hi in place, lo into the buffer
    // right behind it (element-wise, layout-agnostic).  Their own warps and their own barrier per shared-memory
    // stage: a clock64 trace of the one-role version showed the converter chain (gather 200 + TMEM store 160 + dH
    // split 500 + fences, ~1150 clk per K block) AND the issuing thread (twelve MMAs, three commits) both longer than
    // the 768 clk of tensor work.  (Also measured, not kept: a separate ring for the split operand so that landing
    // stages recycle without waiting for the tensor core - 4% slower.)
    const int ct = (warp - 6) * 32 + lane;             // 0..127: share of the dH slab
    for (int kb = 0; kb < num_kb; ++kb) {
      const int s = kb % kStages;
      mbar_wait(full(s), (kb / kStages) & 1);
      const uint32_t ys = base + s * WG_STAGE_BYTES + WG_X_BYTES;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const uint32_t addr = ys + (ct + 128 * u) * 16;
        float4 v;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
        uint32_t h4[4], l4[4];
        split_tf32(v.x, h4[0], l4[0]); split_tf32(v.y, h4[1], l4[1]);
        split_tf32(v.z, h4[2], l4[2]); split_tf32(v.w, h4[3], l4[3]);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(h4[0]), "r"(h4[1]), "r"(h4[2]), "r"(h4[3]) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr + WG_Y_BYTES), "r"(l4[0]), "r"(l4[1]), "r"(l4[2]), "r"(l4[3]) : "memory");
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic writes -> visible to the tensor core
      mbar_arrive(y_ready(s));
    }
  } else {
    // ------------------------------------------------------------ accumulators
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    const int num_chains = (num_kb + kWgChain - 1) / kWgChain;
    for (int chain = 0; chain < num_chains; ++chain) {
      mbar_wait(acc_full, chain & 1);
      tc_fence_after();
      const bool last = chain == num_chains - 1;
#pragma unroll 1
      for (int c0 = 0; c0 < 128; c0 += 32) {
        uint32_t v[32], w[32], run[32];
        tmem_ld32(tmem_base + lane_addr + ACC_MAIN + c0, v);
        tmem_ld32(tmem_base + lane_addr + ACC_CORR + c0, w);
        if (chain > 0) tmem_ld32(tmem_base + lane_addr + RUN_COL + c0, run);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int q = 0; q < 32; ++q) {
          float x = __uint_as_float(v[q]) + __uint_as_float(w[q]);
          if (chain > 0) x += __uint_as_float(run[q]);
          run[q] = __float_as_uint(x);
        }
        if (!last) {
          tmem_st32(tmem_base + lane_addr + RUN_COL + c0, run);
        } else if (i0 + r < k_rows) {                 // rows past K_in exist only as zero-filled TMA padding
          float* op = out + static_cast<int64_t>(i0 + r) * ldo + j0 + c0;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(op + 4 * q) = make_float4(__uint_as_float(run[4 * q]), __uint_as_float(run[4 * q + 1]),
                                                                 __uint_as_float(run[4 * q + 2]), __uint_as_float(run[4 * q + 3]));
        }
      }
      if (!last) {
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        mbar_arrive(acc_empty);
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
  }
}

// ---------------------------------------------------------------------------------------------
// CTA-pair form of the weight gradient (K_in % 256 == 0).  The one-CTA kernel above is bound by shared-memory
// bandwidth: per K block it moves TMA 32 KB + A^T gather 16 KB + dH split 16 KB read / 32 KB written + MMA operand
// reads 48 KB = 144 KB at 128 B/clk = 1125 clk against 768 clk of tensor work (profiles/r01_gemm_kernels.md).  A pair
// computes a 256 x 128 tile of dW: each CTA converts its own 128 columns of the A slab but lands, splits and feeds
// only HALF of the dH slab (64 columns), 88 KB per K block and SM.  Accumulators stay [main | correction] of 128
// columns each (three N = 128 instructions per K step) so that the running sum of the chain folds still fits TMEM.
// Protocol as in linear_tc_pair_kernel: the leader CTA issues, converters / splitters / accumulator warps of both
// CTAs arrive on the leader's barriers (one remote arrive per warp), tcgen05.commit multicasts the releases.
constexpr int kWgPStages = 6;
constexpr uint32_t WGP_Y_BYTES = 32 * 64 * 4;            // 8 KB: this CTA's half of the dH slab (two 32-column boxes)
constexpr uint32_t WGP_STAGE_BYTES = WG_X_BYTES + 2 * WGP_Y_BYTES;   // 32 KB
constexpr uint32_t kWgPSmemBytes = kWgPStages * WGP_STAGE_BYTES + 1024 + 256;
// D = F32, A = B = TF32, A K-major (TMEM), B MN-major, N = 128, M = 256 across the pair
constexpr uint32_t kWgPairDesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | (static_cast<uint32_t>(128 >> 3) << 17) |
                                 (static_cast<uint32_t>(256 >> 4) << 24);

// fp16 variant (kF16): the same pipeline on kind::f16 MMAs, two K = 16 steps per 32-row block instead of four K = 8 steps.
// A^T is packed two rows per 32-bit tensor-memory cell by the converters; the dH half slab lands RAW (one unswizzled
// 32 x 64 fp32 box, 8 KB) and the splitter warps write its fp16 hi / 2^11-scaled lo parts (4 KB each) in the canonical
// MN-major SWIZZLE_128B layout of 16-bit operands: 64 elements (128 B) along N per K row, 8-row groups 1024 B apart, the
// 16-byte chunk index XORed with the row index inside the group.  Operand scales as in linear_tc_pair_kernel<true>.
constexpr uint32_t kWgPairDescH = (1u << 4) | (1u << 16) | (static_cast<uint32_t>(128 >> 3) << 17) | (static_cast<uint32_t>(256 >> 4) << 24);
__device__ __forceinline__ uint64_t make_mnmajor_f16_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>(1024 >> 4) << 16;                    // leading byte offset: next 64 columns (unused: N = 64 per CTA)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                    // stride byte offset: next 8 K rows
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;                            // SWIZZLE_128B
  return d;
}

template <bool kF16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kWgThreads, 1) wgrad_tc_pair_kernel(
    const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_y,
    float* __restrict__ out, int64_t out_split_stride, int ldo, int num_kb_total, int kb_per_split, int kWgChain,
    int k_rows, const float* __restrict__ a_amax, const float* __restrict__ b_amax) {
  extern __shared__ uint8_t smem_dyn[];
  const uint32_t base = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  const uint32_t bars = base + kWgPStages * WGP_STAGE_BYTES;
  auto full = [&](int s) { return bars + 8u * s; };
  auto smem_empty = [&](int s) { return bars + 48u + 8u * s; };
  auto y_ready = [&](int s) { return bars + 96u + 8u * s; };
  auto a_ready = [&](int t) { return bars + 144u + 8u * t; };
  auto a_empty = [&](int t) { return bars + 160u + 8u * t; };
  const uint32_t acc_full = bars + 176u, acc_empty = bars + 184u, tmem_slot = bars + 192u;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = blockIdx.x & 1;
  const int i0 = (blockIdx.x >> 1) * 256 + rank * 128;   // this CTA's rows of dW = its columns of the A slab
  const int j0 = blockIdx.y * 128;
  const int jh = j0 + 64 * rank;                         // this CTA's half of the dH columns
  const int kb_begin = blockIdx.z * kb_per_split;
  const int kb_end = min(num_kb_total, kb_begin + kb_per_split);
  const int num_kb = kb_end - kb_begin;                 // host guarantees >= 1
  out += static_cast<int64_t>(blockIdx.z) * out_split_stride;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_y));
    for (int s = 0; s < kWgPStages; ++s) {
      mbar_init(full(s), 1);
      mbar_init(smem_empty(s), 1);
      mbar_init(y_ready(s), 8);                   // one arrive per splitter warp of both CTAs (leader's copy is used)
    }
    for (int t = 0; t < kWgAStages; ++t) {
      mbar_init(a_ready(t), 8);                   // one arrive per A^T converter warp of both CTAs
      mbar_init(a_empty(t), 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 8);                      // one arrive per accumulator warp of both CTAs
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kWgPStages;
        mbar_wait(smem_empty(s), ((kb / kWgPStages) & 1) ^ 1);
        const uint32_t xs = base + s * WGP_STAGE_BYTES;
        const int m = (kb_begin + kb) * 32;
        mbar_arrive_expect_tx(full(s), WG_X_BYTES + WGP_Y_BYTES);
        tma_load_2d(xs, &map_x, i0, m, full(s));
        tma_load_2d(xs + WG_X_BYTES, &map_y, jh, m, full(s));
        if (!kF16) tma_load_2d(xs + WG_X_BYTES + 4096, &map_y, jh + 32, m, full(s));   // fp16: one raw 32 x 64 box
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      const uint32_t leader = elect_one();
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % kWgPStages, t = kb % kWgAStages;
        const int chain = kb / kWgChain, pos = kb % kWgChain;
        if (pos == 0 && chain > 0) mbar_wait(acc_empty, (chain - 1) & 1);   // accumulators of both CTAs drained
        mbar_wait(a_ready(t), (kb / kWgAStages) & 1);     // A^T of both CTAs is in tensor memory
        mbar_wait(y_ready(s), (kb / kWgPStages) & 1);     // both halves of the dH slab are split
        tc_fence_after();
        if (leader) {
          const uint32_t y_hi = base + s * WGP_STAGE_BYTES + WG_X_BYTES;
          const uint32_t a_hi = tmem_base + A_COL + t * 64;
          if (kF16) {
            const uint64_t d_hi = make_mnmajor_f16_desc(y_hi + WGP_Y_BYTES);          // fp16 hi behind the raw slab, lo behind it
            const uint64_t d_lo = make_mnmajor_f16_desc(y_hi + WGP_Y_BYTES + 4096);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const uint64_t koff = static_cast<uint64_t>((k * 2048) >> 4);          // 16 rows = two 8-row groups per K step
              const uint32_t acc = (pos > 0 || k > 0) ? 1u : 0u;
              mma_f16_ts_pair(tmem_base + ACC_MAIN, a_hi + k * 8, d_hi + koff, kWgPairDescH, acc);
              mma_f16_ts_pair(tmem_base + ACC_CORR, a_hi + k * 8, d_lo + koff, kWgPairDescH, acc);
              mma_f16_ts_pair(tmem_base + ACC_CORR, a_hi + 32 + k * 8, d_hi + koff, kWgPairDescH, 1u);
            }
          } else {
            const uint64_t d_hi = make_mnmajor_b32_desc(y_hi);
            const uint64_t d_lo = make_mnmajor_b32_desc(y_hi + WGP_Y_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t koff = static_cast<uint64_t>((k * 8 * 128) >> 4);       // 8 rows of 128 B per K step
              const uint32_t acc = (pos > 0 || k > 0) ? 1u : 0u;
              mma_tf32_ts_pair(tmem_base + ACC_MAIN, a_hi + k * 8, d_hi + koff, kWgPairDesc, acc);
              mma_tf32_ts_pair(tmem_base + ACC_CORR, a_hi + k * 8, d_lo + koff, kWgPairDesc, acc);
              mma_tf32_ts_pair(tmem_base + ACC_CORR, a_hi + 32 + k * 8, d_hi + koff, kWgPairDesc, 1u);
            }
          }
          tc_commit_pair(smem_empty(s));
          tc_commit_pair(a_empty(t));
          if (pos == kWgChain - 1 || kb == num_kb - 1) tc_commit_pair(acc_full);
        }
        __syncwarp();
      }
    }
  } else if (warp < 6) {
    // ------------------------------------------------------------ A^T converters: column i of the A slab -> TMEM
    const int quarter = warp & 3;
    const int i = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    const float a_scale = kF16 ? f16_scale(__ldg(a_amax)) : 1.f;
    for (int kb = 0; kb < num_kb; ++kb) {
      const int s = kb % kWgPStages, t = kb % kWgAStages;
      mbar_wait(full(s), (kb / kWgPStages) & 1);
      const uint32_t xs = base + s * WGP_STAGE_BYTES;
      uint32_t hi[32], lo[32];
      if (kF16) {
#pragma unroll
        for (int m = 0; m < 16; ++m) {                         // rows 2m, 2m+1 of the slab share one tensor-memory cell
          float v0, v1;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v0) : "r"(xs + ((2 * m) * 128 + i) * 4));
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v1) : "r"(xs + ((2 * m + 1) * 128 + i) * 4));
          split_f16x2(v0 * a_scale, v1 * a_scale, hi[m], lo[m]);
        }
      } else {
#pragma unroll
        for (int m = 0; m < 32; ++m) {
          float v;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(xs + (m * 128 + i) * 4));
          split_tf32(v, hi[m], lo[m]);
        }
      }
      mbar_wait(a_empty(t), ((kb / kWgAStages) & 1) ^ 1);
      tc_fence_after();
      const uint32_t a_hi = tmem_base + lane_addr + A_COL + t * 64;
      if (kF16) {
        tmem_st16(a_hi, *reinterpret_cast<const uint32_t(*)[16]>(hi));
        tmem_st16(a_hi + 32, *reinterpret_cast<const uint32_t(*)[16]>(lo));
      } else {
        tmem_st32(a_hi, hi);
        tmem_st32(a_hi + 32, lo);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(a_ready(t));
    }
  } else if (warp < 10) {
    // ------------------------------------------------------------ dH splitters: this CTA's 64 columns, hi in place,
    // lo into the two boxes right behind
    const int ct = (warp - 6) * 32 + lane;
    const float b_scale = kF16 ? f16_scale(__ldg(b_amax)) : 1.f;
    for (int kb = 0; kb < num_kb; ++kb) {
      const int s = kb % kWgPStages;
      mbar_wait(full(s), (kb / kWgPStages) & 1);
      const uint32_t ys = base + s * WGP_STAGE_BYTES + WG_X_BYTES;
      if (kF16) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int q = ct + 128 * u;                          // 32 rows x 8 chunks of 8 columns
          const int row = q >> 3, ch = q & 7;
          float4 v0, v1;
          const uint32_t src = ys + row * 256 + ch * 32;
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v0.x), "=f"(v0.y), "=f"(v0.z), "=f"(v0.w) : "r"(src));
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v1.x), "=f"(v1.y), "=f"(v1.z), "=f"(v1.w) : "r"(src + 16));
          uint32_t h4[4], l4[4];
          split_f16x2(v0.x * b_scale, v0.y * b_scale, h4[0], l4[0]);
          split_f16x2(v0.z * b_scale, v0.w * b_scale, h4[1], l4[1]);
          split_f16x2(v1.x * b_scale, v1.y * b_scale, h4[2], l4[2]);
          split_f16x2(v1.z * b_scale, v1.w * b_scale, h4[3], l4[3]);
          const uint32_t dst = ys + WGP_Y_BYTES + (row >> 3) * 1024 + (row & 7) * 128 + ((ch ^ (row & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(h4[0]), "r"(h4[1]), "r"(h4[2]), "r"(h4[3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + 4096), "r"(l4[0]), "r"(l4[1]), "r"(l4[2]), "r"(l4[3]) : "memory");
        }
      } else
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t addr = ys + (ct + 128 * u) * 16;
        float4 v;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
        uint32_t h4[4], l4[4];
        split_tf32(v.x, h4[0], l4[0]); split_tf32(v.y, h4[1], l4[1]);
        split_tf32(v.z, h4[2], l4[2]); split_tf32(v.w, h4[3], l4[3]);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(h4[0]), "r"(h4[1]), "r"(h4[2]), "r"(h4[3]) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr + WGP_Y_BYTES), "r"(l4[0]), "r"(l4[1]), "r"(l4[2]), "r"(l4[3]) : "memory");
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic writes -> visible to the tensor cores
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(y_ready(s));
    }
  } else {
    // ------------------------------------------------------------ accumulators (each CTA folds its own 128 rows)
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    const int num_chains = (num_kb + kWgChain - 1) / kWgChain;
    const float out_scale = kF16 ? (1.f / f16_scale(__ldg(a_amax))) * (1.f / f16_scale(__ldg(b_amax))) : 1.f;
    for (int chain = 0; chain < num_chains; ++chain) {
      mbar_wait(acc_full, chain & 1);
      tc_fence_after();
      const bool last = chain == num_chains - 1;
#pragma unroll 1
      for (int c0 = 0; c0 < 128; c0 += 32) {
        uint32_t v[32], w[32], run[32];
        tmem_ld32(tmem_base + lane_addr + ACC_MAIN + c0, v);
        tmem_ld32(tmem_base + lane_addr + ACC_CORR + c0, w);
        if (chain > 0) tmem_ld32(tmem_base + lane_addr + RUN_COL + c0, run);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int q = 0; q < 32; ++q) {
          float x = kF16 ? fmaf(__uint_as_float(w[q]), 1.f / 2048.f, __uint_as_float(v[q])) : __uint_as_float(v[q]) + __uint_as_float(w[q]);
          if (chain > 0) x += __uint_as_float(run[q]);
          if (kF16 && last) x *= out_scale;                    // undo the operand scales (powers of two)
          run[q] = __float_as_uint(x);
        }
        if (!last) {
          tmem_st32(tmem_base + lane_addr + RUN_COL + c0, run);
        } else if (i0 + r < k_rows) {
          float* op = out + static_cast<int64_t>(i0 + r) * ldo + j0 + c0;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(op + 4 * q) = make_float4(__uint_as_float(run[4 * q]), __uint_as_float(run[4 * q + 1]),
                                                                 __uint_as_float(run[4 * q + 2]), __uint_as_float(run[4 * q + 3]));
        }
      }
      if (!last) {
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(acc_empty);
      }
    }
    tc_fence_before();
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols));
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      cudaGetLastError();
  }
  return fn;
}

// 2-D fp32 tensor [rows, inner] with a row pitch of ld elements; box = [box_rows, box_inner].
static int make_map(CUtensorMap* map, const float* ptr, int64_t rows, int64_t inner, int64_t ld, int box_rows,
                    int box_inner = BK, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(GCS_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(inner), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * sizeof(float)};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_inner), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GCS_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(r));
  return GCS_OK;
}

// 2-D fp16 tensor [rows, inner], row pitch ld elements; box = [box_rows, 64] = 128 B rows, SWIZZLE_128B.
static int make_map_f16(CUtensorMap* map, const __half* ptr, int64_t rows, int64_t inner, int64_t ld, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(GCS_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(inner), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * sizeof(__half)};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BKH), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GCS_ERR_CUDA, "cuTensorMapEncodeTiled (fp16) failed with CUresult %d", static_cast<int>(r));
  return GCS_OK;
}

bool shape_ok(int64_t M, int K, int N, const float* A, int64_t lda, const float* C, int64_t ldc, const float* bias) {
  return M > 0 && K % BK == 0 && N % BN == 0 && lda % 4 == 0 && ldc % 4 == 0 && aligned16(A) && aligned16(C) &&
         (!bias || aligned16(bias)) && ceil_div(M, 2 * BM) * (N / BN) < (1LL << 30);
}

int split_strided(const float* W, int rows, int cols, int64_t ldw, bool transpose, int64_t ldo, float* hi, float* lo,
                  cudaStream_t st);

int64_t split_workspace_bytes(int K, int N) { return round_up(2LL * K * N * sizeof(float), 256); }

static int g_max_chain_k_f16 = 1024;                     // ... of the fp16 variant (K = 16 per step: 64 steps; 96 left one hidden-512 gradient tensor 1.3e-5 off)
void set_max_chain_k_f16(int k) { if (k >= BKH && k % BKH == 0) g_max_chain_k_f16 = k; }
static int g_max_chain_k = 768;                          // longest tensor-core accumulation chain of the forward / dX kernel
void set_max_chain_k(int k) { if (k >= BK && k % BK == 0) g_max_chain_k = k; }

// Bt: weights already split, laid out [N][K] (reduction contiguous): hi at Bt, lo at Bt + N*K.
int launch(const float* A, int64_t lda, const float* Bt_hi, const float* Bt_lo, const float* bias, float* C, int64_t ldc,
           int64_t M, int K, int N, int accumulate, cudaStream_t st, const float* rowbias, int64_t ld_rowbias,
           const int64_t* seg) {
  alignas(64) CUtensorMap ma, mh, ml, mc;
  GCS_TRY(make_map(&mc, C, M, N, ldc, 32, 32));        // output boxes of 32 rows x 32 columns (128 B rows, SWIZZLE_128B)
  static bool attr = false;
  if (!attr) {
    GCS_CUDA(cudaFuncSetAttribute(linear_tc_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPSmemBytes));
    attr = true;
  }
  const int n_tiles = N / BN;
  const int num_tiles = static_cast<int>(ceil_div(M, 2 * BM)) * n_tiles;
  const int pairs = num_tiles < sm_count() / 2 ? num_tiles : sm_count() / 2;      // persistent: one CTA pair per SM pair
  dim3 grid(2, pairs);                                                           // x = rank in the pair
  // The tensor core adds every K = 8 step into the fp32 accumulator with TRUNCATION: a chain of n steps shrinks the
  // result by ~n * 2^-26 (measured 2e-5 on the BatchNorm variances of a hidden-512 model with K = 2048 in one chain;
  // with chains of 1024 one gradient tensor of that model was 1.4e-5 off the float64 oracle, with 512 all are inside
  // max(1e-5, 4 x the error of a float32 CPU run), with 768 as well).  Longer reductions therefore run as chunks of
  // <= 768 (96 steps) that meet in C through the epilogue's round-to-nearest reduce-add.
  const int kMaxChainK = g_max_chain_k;
  for (int k0 = 0; k0 < K; k0 += kMaxChainK) {
    const int kc = K - k0 < kMaxChainK ? K - k0 : kMaxChainK;
    GCS_TRY(make_map(&ma, A + k0, M, kc, lda, BM));
    GCS_TRY(make_map(&mh, Bt_hi + k0, N, kc, K, 64));
    GCS_TRY(make_map(&ml, Bt_lo + k0, N, kc, K, 64));
    const bool first = k0 == 0;
    linear_tc_pair_kernel<false><<<grid, kThreads, kPSmemBytes, st>>>(ma, mh, ml, mc, first ? bias : nullptr, M, kc, n_tiles, num_tiles,
                                                                      first ? accumulate : 1, first ? rowbias : nullptr, ld_rowbias,
                                                                      seg, nullptr, nullptr, nullptr, nullptr, nullptr);
    GCS_CHECK_LAUNCH("linear_tc_pair_kernel");
  }
  return GCS_OK;
}

// ---- fp16 variant -------------------------------------------------------------------------------------------------
// Workspace of one GEMM: [hi fp16 N*K | lo fp16 N*K | cells: weights amax, 1/weights scale, scratch A amax] - inside
// split_workspace_bytes(K, N) (the tf32 split needs twice the operand bytes).
static int g_f16 = 1;      // 0 = tf32 kernels only, 1 = fp16 where the caller knows the A operand's |max|, 2 = fp16 everywhere (|max| by an extra pass)
void set_f16_mode(int v) { if (v >= 0 && v <= 2) g_f16 = v; }
int f16_mode() { return g_f16; }
int f16_max_chain() { return g_max_chain_k_f16; }
bool f16_shape_ok(int K) { return K % BKH == 0; }
float* f16_cells(void* workspace, int K, int N) {
  return reinterpret_cast<float*>(static_cast<char*>(workspace) + round_up(4LL * K * N, 256));
}
int64_t f16_workspace_bytes(int K, int N) { return round_up(4LL * K * N, 256) + 256; }

int f16_begin(float* cells, cudaStream_t st) {
  GCS_CUDA(cudaMemsetAsync(cells, 0, 3 * sizeof(float), st));
  return GCS_OK;
}
int absmax(const float* A, int64_t lda, int64_t M, int K, float* cell, cudaStream_t st, const float* col_scale) {
  int64_t blocks = M < 8LL * sm_count() ? M : 8LL * sm_count();
  if (blocks < 1) blocks = 1;
  absmax_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(A, lda, M, K, cell, col_scale);
  GCS_CHECK_LAUNCH("absmax_kernel");
  return GCS_OK;
}
int fold_bias(const float* bias, const float* scale, const float* shift, int N, float* out, cudaStream_t st) {
  fold_bias_kernel<<<static_cast<unsigned>(ceil_div(N, 128)), 128, 0, st>>>(bias, scale, shift, N, out);
  GCS_CHECK_LAUNCH("fold_bias_kernel");
  return GCS_OK;
}
int amax_merge(float* cell, const float* other, cudaStream_t st) {
  amax_merge_kernel<<<1, 1, 0, st>>>(cell, other);
  GCS_CHECK_LAUNCH("amax_merge_kernel");
  return GCS_OK;
}
int split_f16_strided(const float* W, int rows, int cols, int64_t ldw, bool transpose, int64_t ldo, void* hi, void* lo,
                      float* cells, cudaStream_t st, const float* col_scale) {
  const int64_t n = static_cast<int64_t>(rows) * cols;
  int64_t blocks = ceil_div(n, 256);
  if (blocks > 4LL * sm_count()) blocks = 4LL * sm_count();
  split_weights_f16_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(W, rows, cols, ldw, transpose ? 1 : 0, ldo,
                                                                        static_cast<__half*>(hi), static_cast<__half*>(lo),
                                                                        cells, cells + 1, col_scale);
  GCS_CHECK_LAUNCH("split_weights_f16_kernel");
  return GCS_OK;
}

// Batched form of absmax + split_f16_strided over n jobs; every job's cells must have been zeroed (the caller clears the
// whole region the jobs live in with one memset).
int split_f16_multi(const SplitJobs& jobs, cudaStream_t st) {
  if (jobs.n <= 0) return GCS_OK;
  if (jobs.n > kMaxSplitJobs) return fail(GCS_ERR_INVALID_ARGUMENT, "split_f16_multi: too many jobs");
  const dim3 grid(96, static_cast<unsigned>(jobs.n));
  absmax_multi_kernel<<<grid, 256, 0, st>>>(jobs);
  GCS_CHECK_LAUNCH("absmax_multi_kernel");
  split_weights_f16_multi_kernel<<<grid, 256, 0, st>>>(jobs);
  GCS_CHECK_LAUNCH("split_weights_f16_multi_kernel");
  return GCS_OK;
}

// Bt: fp16 split weights [N][K] (hi, lo), cells as left by split_f16_strided; a_amax: device |max| of A.
int launch_f16(const float* A, int64_t lda, const void* Bt_hi, const void* Bt_lo, const float* cells, const float* a_amax,
               const float* bias, float* C, int64_t ldc, int64_t M, int K, int N, int accumulate, cudaStream_t st,
               const float* rowbias, int64_t ld_rowbias, const int64_t* seg, const float* alpha, float* amax_out,
               float* stats_part) {
  if ((alpha || amax_out || stats_part) && K > g_max_chain_k_f16)
    return fail(GCS_ERR_UNSUPPORTED, "launch_f16: the PReLU / |max| / statistics epilogue needs the reduction in one chain");
  alignas(64) CUtensorMap ma, mh, ml, mc;
  const __half* bh = static_cast<const __half*>(Bt_hi);
  const __half* bl = static_cast<const __half*>(Bt_lo);
  // chains as in launch(): a K = 16 step adds into the accumulator with the same truncation, half as many steps per K
  const int kMaxChainK = g_max_chain_k_f16;
  if (N % 256 == 0) {
    // one pass over A per 256 output columns (linear_f16_pass256_kernel); output boxes of 32 rows x 16 columns
    GCS_TRY(make_map(&mc, C, M, N, ldc, 32, 16, CU_TENSOR_MAP_SWIZZLE_64B));
    static bool attr256 = false;
    if (!attr256) {
      GCS_CUDA(cudaFuncSetAttribute(linear_f16_pass256_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSSmemBytes));
      attr256 = true;
    }
    const int num_tiles = static_cast<int>(ceil_div(M, 2 * BM)) * (N / 256);
    const int pairs = num_tiles < sm_count() / 2 ? num_tiles : sm_count() / 2;
    dim3 grid(2, pairs);
    for (int k0 = 0; k0 < K; k0 += kMaxChainK) {
      const int kc = K - k0 < kMaxChainK ? K - k0 : kMaxChainK;
      GCS_TRY(make_map(&ma, A + k0, M, kc, lda, BM));
      GCS_TRY(make_map_f16(&mh, bh + k0, N, kc, K, 128));
      GCS_TRY(make_map_f16(&ml, bl + k0, N, kc, K, 128));
      const bool first = k0 == 0;
      linear_f16_pass256_kernel<<<grid, kHThreads, kSSmemBytes, st>>>(ma, mh, ml, mc, first ? bias : nullptr, M, kc, N, num_tiles,
                                                                       first ? accumulate : 1, first ? rowbias : nullptr, ld_rowbias,
                                                                       seg, a_amax, cells + 1, alpha, amax_out, stats_part);
      GCS_CHECK_LAUNCH("linear_f16_pass256_kernel");
    }
    return GCS_OK;
  }
  GCS_TRY(make_map(&mc, C, M, N, ldc, 32, 32));
  static bool attr = false;
  if (!attr) {
    GCS_CUDA(cudaFuncSetAttribute(linear_tc_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kHSmemBytes));
    attr = true;
  }
  const int n_tiles = N / BN;
  const int num_tiles = static_cast<int>(ceil_div(M, 2 * BM)) * n_tiles;
  const int pairs = num_tiles < sm_count() / 2 ? num_tiles : sm_count() / 2;
  dim3 grid(2, pairs);
  for (int k0 = 0; k0 < K; k0 += kMaxChainK) {
    const int kc = K - k0 < kMaxChainK ? K - k0 : kMaxChainK;
    GCS_TRY(make_map(&ma, A + k0, M, kc, lda, BM));
    GCS_TRY(make_map_f16(&mh, bh + k0, N, kc, K, 64));
    GCS_TRY(make_map_f16(&ml, bl + k0, N, kc, K, 64));
    const bool first = k0 == 0;
    linear_tc_pair_kernel<true><<<grid, kHThreads, kHSmemBytes, st>>>(ma, mh, ml, mc, first ? bias : nullptr, M, kc, n_tiles, num_tiles,
                                                                     first ? accumulate : 1, first ? rowbias : nullptr, ld_rowbias,
                                                                     seg, a_amax, cells + 1, alpha, amax_out, stats_part);
    GCS_CHECK_LAUNCH("linear_tc_pair_kernel<f16>");
  }
  return GCS_OK;
}

bool wgrad_shape_ok(int64_t M, int K, int N, const float* A, int64_t lda, const float* dH, int64_t ldh) {
  // K_in < 128 (the first layer: raw features, all positive against a zero-sum dH) stays on the exact
  // FFMA path: measured 2.1e-5 gradient error there with the truncating tensor-core accumulation.
  return M > 0 && K % 128 == 0 && N % 128 == 0 && lda % 4 == 0 && ldh % 4 == 0 && aligned16(A) && aligned16(dH) &&
         M < (1LL << 31) - 64;
}

static int g_wg_f16 = 1;                                 // debug knob (gcs_debug_set_param 9): 0 = weight gradient on the tf32 split only
void set_wgrad_f16(int v) { g_wg_f16 = v; }
static int g_wg_pair = 1;                                // debug knob: 0 = always the one-CTA kernel
void set_wgrad_pair(int v) { g_wg_pair = v; }
static bool wgrad_use_pair(int K) { return g_wg_pair && K % 256 == 0; }

// Number of row splits (grid.z) and K blocks per split for the weight-gradient kernel.
void wgrad_split(int64_t M, int K, int N, int* splits, int* kb_per_split) {
  const int64_t nkb = ceil_div(M, 32);
  const int kWgChain = g_wg_chain;
  const int64_t max_s = ceil_div(nkb, kWgChain);          // at least one full chain per split
  int64_t s;
  if (wgrad_use_pair(K)) {
    const int64_t tiles = (K / 256) * (N / 128);          // 256 x 128 tiles, one CTA pair each: ONE wave of pairs
    s = (sm_count() / 2) / tiles;
  } else {
    const int64_t tiles = ceil_div(K, 128) * (N / 128);
    s = ceil_div(4LL * sm_count(), tiles);
  }
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  int64_t per = ceil_div(nkb, s);
  per = round_up(per, kWgChain);                           // whole chains except in the last split
  *kb_per_split = static_cast<int>(per);
  *splits = static_cast<int>(ceil_div(nkb, per));
}

int64_t wgrad_workspace_bytes(int64_t M, int K, int N) {
  int s, per;
  wgrad_split(M, K, N, &s, &per);
  return round_up(static_cast<int64_t>(s) * K * N * sizeof(float), 256);
}

// partials: [splits][K][N]; with one split the result goes straight to dW (ld = N).
bool wgrad_f16_ok(int K) { return g_f16 != 0 && g_wg_f16 != 0 && wgrad_use_pair(K); }

// a_amax / b_amax: device |max| of A and dH (both or neither): the fp16 variant of the pair kernel.
int wgrad_launch(const float* A, int64_t lda, const float* dH, int64_t ldh, float* out, int64_t M, int K, int N,
                 int splits, int kb_per_split, cudaStream_t st, const float* a_amax, const float* b_amax) {
  alignas(64) CUtensorMap mx, my;
  GCS_TRY(make_map(&mx, A, M, K, lda, 32, 128, CU_TENSOR_MAP_SWIZZLE_NONE));
  const bool f16 = a_amax && b_amax && wgrad_f16_ok(K);
  if (f16) GCS_TRY(make_map(&my, dH, M, N, ldh, 32, 64, CU_TENSOR_MAP_SWIZZLE_NONE));      // raw 32 x 64 slab halves
  else GCS_TRY(make_map(&my, dH, M, N, ldh, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
  if (wgrad_use_pair(K)) {
    static bool attr2 = false;
    if (!attr2) {
      GCS_CUDA(cudaFuncSetAttribute(wgrad_tc_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgPSmemBytes));
      GCS_CUDA(cudaFuncSetAttribute(wgrad_tc_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgPSmemBytes));
      attr2 = true;
    }
    dim3 grid(static_cast<unsigned>(2 * (K / 256)), N / 128, splits);       // x = 2 * tile + rank in the pair
    if (f16)
      wgrad_tc_pair_kernel<true><<<grid, kWgThreads, kWgPSmemBytes, st>>>(mx, my, out, static_cast<int64_t>(K) * N, N,
                                                                        static_cast<int>(ceil_div(M, 32)), kb_per_split,
                                                                        g_wg_chain, K, a_amax, b_amax);
    else
      wgrad_tc_pair_kernel<false><<<grid, kWgThreads, kWgPSmemBytes, st>>>(mx, my, out, static_cast<int64_t>(K) * N, N,
                                                                         static_cast<int>(ceil_div(M, 32)), kb_per_split,
                                                                         g_wg_chain, K, nullptr, nullptr);
    GCS_CHECK_LAUNCH("wgrad_tc_pair_kernel");
    return GCS_OK;
  }
  static bool attr = false;
  if (!attr) {
    GCS_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmemBytes));
    attr = true;
  }
  dim3 grid(static_cast<unsigned>(ceil_div(K, 128)), N / 128, splits);
  wgrad_tc_kernel<<<grid, kWgThreads, kWgSmemBytes, st>>>(mx, my, out, static_cast<int64_t>(K) * N, N,
                                                         static_cast<int>(ceil_div(M, 32)), kb_per_split, g_wg_chain, K);
  GCS_CHECK_LAUNCH("wgrad_tc_kernel");
  return GCS_OK;
}

int split(const float* W, int rows, int cols, bool transpose, float* hi, float* lo, cudaStream_t st) {
  return split_strided(W, rows, cols, cols, transpose, transpose ? rows : cols, hi, lo, st);
}

int split_strided(const float* W, int rows, int cols, int64_t ldw, bool transpose, int64_t ldo, float* hi, float* lo,
                  cudaStream_t st) {
  const int64_t n = static_cast<int64_t>(rows) * cols;
  int64_t blocks = ceil_div(n, 256);
  if (blocks > 4LL * sm_count()) blocks = 4LL * sm_count();
  split_weights_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(W, rows, cols, ldw, transpose ? 1 : 0, ldo, hi, lo);
  GCS_CHECK_LAUNCH("split_weights_kernel");
  return GCS_OK;
}

}  // namespace tc
}  // namespace gcs
