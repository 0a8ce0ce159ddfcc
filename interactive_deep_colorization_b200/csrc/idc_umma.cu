// tcgen05 engine: implicit-GEMM convolution on the 5th-gen tensor cores (sm_100a).
//
//   D[128 pixels x BN couts] (FP32, TMEM) += A[128 x 64] (smem, K-major, SW128) * B[BN x 64]^T
//
// * A tiles are gathered by TMA straight from the NHWC activation planes: one 4-D box
//   {64 ch, wbox, hbox, 1 image} per filter tap, shifted by the tap offset; out-of-bounds
//   pixels are zero-filled by TMA (= the reference's zero padding), the `::2` decimation
//   (model.py:149-151) and the output-parity views of the transposed convs are expressed as
//   tensor-map strides, so no im2col / decimated copy ever exists in HBM.
// * 1e-3 ab parity needs ~22 mantissa bits (SURVEY 7.3): activations and weights are stored as
//   FP16 hi + lo planes and every product is issued as 3 MMAs (hi*hi + hi*lo + lo*hi) into the
//   same FP32 TMEM accumulator.  IDC_FLAG_FAST_FP16 drops the lo planes (1 MMA).
// * The tensor core's FP32 accumulator does not round to nearest: measured on B200 (round 1), a
//   K=4608 layer accumulated entirely in TMEM (864 MMA steps) loses ~1e-5 relative per layer and the
//   network ends at 1.2e-2 ab error although all three split terms are present.  So accumulation
//   is CHUNKED: the tensor core only sums `chunk_kb` k-blocks (default 1 = 12 MMAs, the 8 small
//   cross terms first) into a fresh TMEM buffer; the accumulate warps add each chunk into FP32
//   REGISTERS with round-to-nearest CUDA-core adds while the next chunk runs (NBUF TMEM buffers).
// * warp roles: warp0 = TMA producer, warp1 = MMA issuer (+TMEM alloc), warps2-9 = accumulate +
//   epilogue (TMEM chunk -> regs += ; at tile end bias/act/BN/global-hints -> hi/lo split -> NHWC
//   store, or the fused model_out head).  Warp w owns TMEM lane quarter w%4 and column half (w-2)/4.
//   Persistent grid = min(tiles, #SM).
// * also in this file: CTA pairs (cta_group::2), the halo-tile A operand, deterministic split-K for launches that
//   cannot fill the machine (128-column tiles; the CTA's own pieces never leave its registers) and
//   conv1_1_umma_kernel (model1.0 as one padded k-block whose operand rows the threads write themselves).
#include <stdio.h>
#include <stdlib.h>

#include "idc_internal.h"

#ifndef IDC_CTA_COUNTERS
#define IDC_CTA_COUNTERS 0   // 1: per-CTA cycle counters for tools/cta_counters.py (costs a few % in the hot loops)
#endif

namespace idc {

constexpr int kBM = 128;      // pixels per tile (UMMA M)
constexpr int kBK = 64;       // channels per k-block (128 bytes of FP16 = one SW128 row)
constexpr int kThreads = 384;   // control warpgroup (TMA, MMA, 2 idle warps) + 2 accumulate/epilogue warpgroups
constexpr int kCtrlRegs = 56;    // setmaxnreg budgets: the control warpgroup gives its registers to the accumulate warps
constexpr int kAccRegs = 224;
constexpr int kAccThreads = 256;

struct UmmaParams {
  const CUtensorMap* amaps;  // device array, [view][hi, lo]
  const int4* kblk;          // [ncls][nkb] : {map index (hi), c0, dy, dx}
  int nkb, ncls;
  int chunk_kb;              // k-blocks accumulated inside the tensor core per chunk (>=1)
  int split_k;               // >1: K is split over `split_k` CTAs per tile (small-batch latency path)
  float* ws;                 // split-K partial sums [work item][128 rows][MT*BN] FP32
  int* counters;             // split-K arrival counters [tile] (self-resetting)
  int n_img, tiles_y, tiles_x, n_tiles_n, total_tiles;
  int hbox, wbox, wshift;
  int Hl, Wl, cout_pad;
  const float* bias;   // bias / descale
  const float* scale;  // bn_scale * descale
  const float* shift;
  const float* gadd;   // [n_img][gadd_ld] or null
  int gadd_ld;
  float gadd_mult;     // output activation scale (2^kActScaleLog2) applied to the global-hints vector
  int act;
  __half* out_hi;
  __half* out_lo;
  int Hout, Wout, Cout, os;
  float* out_f32;      // logits [M][out_ld] or null
  int out_ld;
  const float* wout;   // fused head weights [2][128] or null
  const float* bout;
  float* out_ab;
  float out_mult;
  int* err;
  long long* dbgbuf;   // experiments only: per-CTA cycle counters [grid][8]
  int n_amaps;         // entries of `amaps` (prefetched in the prologue)
  int max_ctas;        // host side only: grid cap for side-branch launches
  int halo_groups;     // HALO kernels: 64-channel input groups (K = 9 taps x halo_groups k-blocks); kblk = {-, B k-column, dy+1, dx+1}
  int img0;            // first image of this launch (n_img = img0 + images of the launch): idc_forward_host
                       // runs the last op in image chunks so that the D2H of a chunk overlaps the next one
};

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug becomes an error code + trap instead of a hung GPU.
__device__ __noinline__ void mbar_timeout(int* err, int code) {
  if (err) {
    atomicExch(err, code);
    __threadfence_system();
  }
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 6000000000LL) mbar_timeout(err, code);
  }
}

// one lane of a converged warp (warp-uniform control flow keeps descriptors / addresses in uniform
// registers; a role wrapped in `if (lane == 0)` makes ptxas re-broadcast every operand per instruction)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// Programmatic dependent launch (PDL): a kernel launched with the programmatic-stream-serialization attribute may
// start while its predecessor is still running; everything that depends on the predecessor's output sits behind
// pdl_wait().  Every thread of every kernel of a forward executes pdl_wait() before it exits, so "kernel k is
// complete" implies "kernels 0..k-1 are complete" (completion stays transitive along the chain).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void prefetch_tmap(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}

// Read-only epilogue vectors: NOT volatile, so ptxas/nvcc may batch the loads of a slab ahead of its math (the
// accumulate warps run 2 per scheduler and cannot hide a serialised ld.shared -> FFMA chain).  `addr` must be
// derived from an epi_token() issued after the staging barrier, which pins the loads below that barrier.
__device__ __forceinline__ float4 ld_shared_f4(uint32_t addr) {
  float4 v;
  asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t epi_token(uint32_t addr) {
  uint32_t r;
  asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(addr) : "memory");
  return r;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// ---- CTA pairs (cta_group::2): the leader (cluster rank 0) issues M=256 MMAs over both SMs; each CTA loads its
//      own 128 pixel rows of A and HALF of the weight tile, so every SM reads 8 KB of operands per MMA
//      instead of 12 KB and the weight tile crosses L2->SM once per pair.  Protocol after DeepGEMM/CUTLASS:
//      TMA (cta_group::2) signals the leader's `full` barrier, tcgen05.commit multicasts to both CTAs'
//      `empty` / `tfull` barriers, the accumulate warps of both CTAs arrive on the leader's `tempty`. ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_rank0(uint32_t local_bar) {   // arrive on the SAME barrier of cluster rank 0
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, 0;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(local_bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, int c2,
                                                 int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {          // arrives on `bar` in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled operand tile: rows of 64 FP16 (128 B), 8-row swizzle atoms 1024 B
// apart (SBO); LBO unused for a single K atom.  Bit layout = cute::UMMA::SmemDescriptor.
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr, uint32_t sbo = 1024u) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);  // start address
  d |= (uint64_t)(sbo >> 4) << 32;              // stride byte offset (pitch of the 8-row groups)
  d |= (uint64_t)1 << 46;                       // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                       // SWIZZLE_128B
  return d;
}
// kind::f16 instruction descriptor: A=B=F16, D=F32, both K-major, M=128, N=BN.
__host__ __device__ constexpr uint32_t make_idesc(int bn, int m = kBM) {
  return (1u << 4) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// two floats -> packed f16x2 (low half = a), saturating to +-65504 instead of inf (one F2FP instruction)
__device__ __forceinline__ uint32_t pack_f16x2_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

// 32 FP32 values -> 16 packed f16x2 words of the hi plane (+ 16 of the lo plane = value - hi, when SPLIT)
template <bool SPLIT>
__device__ __forceinline__ void split_pack(const float (&f)[32], uint32_t (&hw)[16], uint32_t (&lw)[16]) {
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    hw[j] = pack_f16x2_sat(f[2 * j], f[2 * j + 1]);
    if (SPLIT) {
      const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hw[j]));
      lw[j] = pack_f16x2_sat(f[2 * j] - hf.x, f[2 * j + 1] - hf.y);
    }
  }
}

__device__ __forceinline__ void split_h(float v, __half& hi, __half& lo) {
  v = fminf(fmaxf(v, -65504.f), 65504.f);
  hi = __float2half_rn(v);
  lo = __float2half_rn(v - __half2float(hi));
}

// HALO (stride-1 3x3 layers): instead of one TMA box per filter tap, ONE halo tile of 18 rows x 10 pixels per
// 64-channel input group serves all 9 taps of a 16-row x 8-pixel M-tile -- the MMA's A descriptor starts at the
// pixel-shifted window (start = slot + ((dy+1)*10 + dx+1)*128 B, SBO = 10*128 B; the 128-byte swizzle is a function
// of the absolute smem address: tools/experiments/halo_desc_probe.cu).  The stage ring then holds weight tiles only.
constexpr int kHaloW = 10, kHaloH = 18;
constexpr int kHaloPlane = (kHaloW * kHaloH * 128 + 1023) / 1024 * 1024;   // 23040 -> 23552
template <int BN, int MT, int CG, bool SPLIT, bool HALO = false>
struct SmemPlan {
  static constexpr int kABytes = MT * kBM * kBK * 2;            // MT M-tiles of 128 pixels x 64 ch FP16 (16 KB each)
  static constexpr int kAStage = HALO ? 0 : kABytes;           // A bytes inside a ring stage (one plane)
  static constexpr int kBBytes = (BN / CG) * kBK * 2;          // CG == 2: each CTA of the pair holds half of the weight tile
  static constexpr int kStageBytes = (SPLIT ? 2 : 1) * (kAStage + kBBytes);
  static constexpr int kHaloSlot = (SPLIT ? 2 : 1) * kHaloPlane;
  static constexpr int kHaloBytes = HALO ? 2 * kHaloSlot : 0;   // two halo slots (double buffered)
  static_assert(!HALO || MT == 1, "halo tiles are single 16x8-pixel M-tiles");
  static constexpr int kTail = 3 * BN * 4 + 272 * 4 + 256 + 128 * 2 * 4;  // epi vecs, head, barriers, head reduce
  static constexpr int kOutStage = 16384;                         // epilogue staging: one private 2 KB transpose tile per accumulate warp
  static constexpr int kBudget = 232448 - 1024 - kTail - kOutStage - kHaloBytes;  // 227 KB opt-in limit minus alignment slack
  static constexpr int kStages = kBudget / kStageBytes >= 4 ? 4 : kBudget / kStageBytes;
  static constexpr int kTotal = kStages * kStageBytes + kHaloBytes + kOutStage + kTail + 1024;   // + alignment slack
  static constexpr int kBufCols = MT * BN;                       // TMEM columns of one chunk buffer
  static constexpr int kNBuf = (512 / kBufCols) >= 4 ? 4 : (512 / kBufCols);
  static constexpr int kTmemCols = (kNBuf * kBufCols <= 128) ? 128 : (kNBuf * kBufCols <= 256 ? 256 : 512);
  static constexpr int kCH = (MT == 2) ? BN : BN / 2;            // accumulator columns per accumulate thread
  static_assert(kStages >= 2, "need at least a double-buffered operand ring");
  static_assert(CG == 1 || BN == 256 || BN == 128 || BN == 64, "pairs: BN/2 weight rows per CTA must be a whole number of swizzle atoms");
};

// ------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------
// The body of umma_conv_kernel.  It stays a separate inlined function: written directly as the __global__ function's
// body, ptxas allocates <128, 2, 2, false> with 24 B of stack and 48 B of spill stores instead of 16 B and 36 B.
template <int BN, int MT, int CG, bool SPLIT, bool HALO>
__device__ __forceinline__ void conv_body(const CUtensorMap& bmap_hi, const CUtensorMap& bmap_lo, const UmmaParams& p) {
  using SP = SmemPlan<BN, MT, CG, SPLIT, HALO>;
  constexpr int STAGES = SP::kStages;
  constexpr bool PAIR = CG == 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_halo = smem + STAGES * SP::kStageBytes;             // HALO: 2 slots x {hi, lo} planes, 1024-aligned
  uint8_t* s_out = s_halo + SP::kHaloBytes;                      // 1024-aligned (stage / plane sizes are multiples of 1 KB)
  uint8_t* tail = s_out + SP::kOutStage;
  float* s_bias = reinterpret_cast<float*>(tail);
  float* s_scale = s_bias + BN;
  float* s_shift = s_scale + BN;
  float* s_head = s_shift + BN;                                   // [2][128] + bias[2] (+pad)
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_head + 272);
  constexpr int NBUF = SP::kNBuf;
  uint64_t* full_bar = s_bar;                      // [STAGES] TMA -> MMA
  uint64_t* empty_bar = s_bar + STAGES;            // [STAGES] MMA -> TMA
  uint64_t* tfull_bar = s_bar + 2 * STAGES;        // [NBUF]   MMA -> accumulate warps (chunk ready)
  uint64_t* tempty_bar = s_bar + 2 * STAGES + NBUF;  // [NBUF] accumulate warps -> MMA (chunk drained)
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 2 * STAGES + 2 * NBUF);
  uint64_t* afull_bar = s_bar + 20;                // [2] HALO: halo TMA -> MMA
  uint64_t* aempty_bar = s_bar + 22;               // [2] HALO: MMA -> halo TMA
  float* s_red = reinterpret_cast<float*>(s_bar + 32);   // [128][2] fused-head partial sums, after the 256-byte barrier block

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long t_kernel0 = (IDC_CTA_COUNTERS && p.dbgbuf) ? clock64() : 0;

  // ---- one-time setup ----
  if (p.wout) {
    for (int i = threadIdx.x; i < 256; i += kThreads) s_head[i] = p.wout[i];
    if (threadIdx.x < 2) s_head[256 + threadIdx.x] = p.bout[threadIdx.x];
  }
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;
  if (threadIdx.x == 32) {                          // descriptors are input-independent: fetch them during the prologue
    prefetch_tmap(&bmap_hi);
    if (SPLIT) prefetch_tmap(&bmap_lo);
    for (int i = 0; i < p.n_amaps; ++i) prefetch_tmap(p.amaps + i);
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), CG);        // pairs: both producers arrive on the leader's barrier
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int a = 0; a < NBUF; ++a) {
      mbar_init(smem_u32(&tfull_bar[a]), 1);
      mbar_init(smem_u32(&tempty_bar[a]), 8 * CG);  // one arrive per accumulate warp (of both CTAs on the leader)
    }
    if (HALO)
      for (int a = 0; a < 2; ++a) {
        mbar_init(smem_u32(&afull_bar[a]), CG);
        mbar_init(smem_u32(&aempty_bar[a]), 1);
      }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // Both CTAs of a pair are running before either executes the cta_group::2 TMEM allocation (it writes the base address
  // into the peer's shared memory too).  Without this barrier results stay bit-identical and a click gets 3 us shorter,
  // but compute-sanitizer's racecheck then reports the allocation -- so it stays.
  if (PAIR) cluster_sync_all();
  if (warp == 1) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                   "r"((uint32_t)SP::kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)),
                   "r"((uint32_t)SP::kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  pdl_launch_dependents();                           // the next kernel of the forward may start its own prologue
  if (warp != 0) pdl_wait();                         // warp 0 first requests its weight tiles (see the producer)

  long long t_wait_tfull_g = 0, t_drain_g = 0, t_epi_g = 0, t_splitk_g = 0, t_spin_g = 0;

  if (warp < 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kCtrlRegs));
  if (warp == 0) {
    // =============================== TMA producer ===============================
    {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t hcount = 0;                               // HALO: halo loads issued (slot = hcount & 1)
      const int tiles_per_img = p.tiles_y * p.tiles_x;
      const int S = p.split_k;
      // Weights never depend on the previous layer: request the weight tiles of this CTA's first k-blocks BEFORE
      // pdl_wait, so they stream in while the predecessor drains.  The stage's `full` barrier is armed with the byte
      // count of the whole stage; the activation boxes follow after the wait.
      const int w0 = blockIdx.x / CG;
      int npre = 0;
      if (w0 < p.total_tiles * S) {
        const int tile = w0 / S, ks = w0 - tile * S;
        const int kbeg = (ks * p.nkb) / S, kend = ((ks + 1) * p.nkb) / S;
        int r = tile;
        const int nt = r % p.n_tiles_n;
        r /= p.n_tiles_n;
        const int cls = r % p.ncls;
        const int brow = cls * p.cout_pad + nt * BN + (int)cta_rank * (BN / CG);
        const int4* kb = p.kblk + cls * p.nkb;
        npre = kend - kbeg < STAGES ? kend - kbeg : STAGES;
        for (int i = 0; i < npre; ++i) {                  // the ring is still empty: k-block kbeg + i goes to stage i
          if (elect_one()) {
            const uint32_t fb = smem_u32(&full_bar[i]);
            const uint32_t sb = smem_u32(smem + i * SP::kStageBytes) + (SPLIT ? 2 : 1) * SP::kAStage;
            const int kcol = HALO ? __ldg(kb + kbeg + i).y : (kbeg + i) * kBK;
            if (PAIR) {
              if (leader) mbar_expect_tx(fb, 2 * SP::kStageBytes); else mbar_arrive_rank0(fb);
              tma_load_2d_pair(sb, &bmap_hi, fb, kcol, brow);
              if (SPLIT) tma_load_2d_pair(sb + SP::kBBytes, &bmap_lo, fb, kcol, brow);
            } else {
              mbar_expect_tx(fb, SP::kStageBytes);
              tma_load_2d(sb, &bmap_hi, fb, kcol, brow);
              if (SPLIT) tma_load_2d(sb + SP::kBBytes, &bmap_lo, fb, kcol, brow);
            }
          }
          __syncwarp();
        }
      }
      pdl_wait();                                       // activations of the previous layer are complete and visible
      for (int w = w0; w < p.total_tiles * S; w += gridDim.x / CG) {
        const int tile = w / S, ks = w - tile * S;
        const int kbeg = (ks * p.nkb) / S, kend = ((ks + 1) * p.nkb) / S;
        const int kpre = (w == w0) ? kbeg + npre : kbeg;        // k-blocks below kpre already have their weight tile
        // tile order: n-tile fastest, then output-parity class, then spatial tile, then image -- CTAs that
        // run together share the A tile (all n-tiles) and the source rows (all 4 classes of an up-layer).
        // Pairs: `tile` counts M-tile PAIRS; this CTA takes M-tile 2*pair + rank.
        int r = tile;
        const int nt = r % p.n_tiles_n;
        r /= p.n_tiles_n;
        const int cls = r % p.ncls;
        r /= p.ncls;
        if (PAIR) r = 2 * r + (int)cta_rank;
        const int img_rel = r / tiles_per_img;
        r -= img_rel * tiles_per_img;
        const int img = p.img0 + img_rel;
        const int y0 = (r / p.tiles_x) * (p.hbox * MT), x0 = (r % p.tiles_x) * p.wbox;
        const int brow = cls * p.cout_pad + nt * BN + (int)cta_rank * (BN / CG);
        const int4* kb = p.kblk + cls * p.nkb;                  // read-only table in global memory (L1-resident)
        if (HALO) {
          // k-block i = (input group i / 9, tap i % 9): one halo load per group, one weight tile per k-block
          for (int k = kbeg; k < kend; ++k) {
            if (k % 9 == 0) {
              const uint32_t slot = hcount & 1, hphase = (hcount >> 1) & 1;
              ++hcount;
              mbar_wait(smem_u32(&aempty_bar[slot]), hphase ^ 1, p.err, 6);
              if (elect_one()) {
                const uint32_t fa = smem_u32(&afull_bar[slot]);
                const uint32_t sh = smem_u32(s_halo + slot * SP::kHaloSlot);
                const int c0 = (k / 9) * kBK;
                constexpr uint32_t kHaloTx = (SPLIT ? 2 : 1) * kHaloW * kHaloH * 128;
                if (PAIR) {
                  if (leader) mbar_expect_tx(fa, 2 * kHaloTx); else mbar_arrive_rank0(fa);
                  tma_load_4d_pair(sh, p.amaps, fa, c0, x0 - 1, y0 - 1, img);
                  if (SPLIT) tma_load_4d_pair(sh + kHaloPlane, p.amaps + 1, fa, c0, x0 - 1, y0 - 1, img);
                } else {
                  mbar_expect_tx(fa, kHaloTx);
                  tma_load_4d(sh, p.amaps, fa, c0, x0 - 1, y0 - 1, img);
                  if (SPLIT) tma_load_4d(sh + kHaloPlane, p.amaps + 1, fa, c0, x0 - 1, y0 - 1, img);
                }
              }
              __syncwarp();
            }
            mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1, p.err, 1);
            if (k >= kpre && elect_one()) {
              const uint32_t fb = smem_u32(&full_bar[stage]);
              const int4 e = __ldg(kb + k);
              const uint32_t sb = smem_u32(smem + stage * SP::kStageBytes);
              if (PAIR) {
                if (leader) mbar_expect_tx(fb, 2 * SP::kStageBytes); else mbar_arrive_rank0(fb);
                tma_load_2d_pair(sb, &bmap_hi, fb, e.y, brow);
                if (SPLIT) tma_load_2d_pair(sb + SP::kBBytes, &bmap_lo, fb, e.y, brow);
              } else {
                mbar_expect_tx(fb, SP::kStageBytes);
                tma_load_2d(sb, &bmap_hi, fb, e.y, brow);
                if (SPLIT) tma_load_2d(sb + SP::kBBytes, &bmap_lo, fb, e.y, brow);
              }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
        if (!HALO)
        for (int k = kbeg; k < kend; ++k) {
          mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1, p.err, 1);
          if (elect_one()) {
            const uint32_t fb = smem_u32(&full_bar[stage]);
            const int4 e = __ldg(kb + k);
            const uint32_t sa = smem_u32(smem + stage * SP::kStageBytes);
            const CUtensorMap* am = p.amaps + e.x;
            const uint32_t sb = sa + (SPLIT ? 2 : 1) * SP::kABytes;
            const bool need_b = k >= kpre;
            if (PAIR) {
              // every byte of both CTAs lands on the LEADER's barrier
              if (need_b) { if (leader) mbar_expect_tx(fb, 2 * SP::kStageBytes); else mbar_arrive_rank0(fb); }
              tma_load_4d_pair(sa, am, fb, e.y, x0 + e.w, y0 + e.z, img);
              if (SPLIT) tma_load_4d_pair(sa + SP::kABytes, am + 1, fb, e.y, x0 + e.w, y0 + e.z, img);
              if (need_b) {
                tma_load_2d_pair(sb, &bmap_hi, fb, k * kBK, brow);
                if (SPLIT) tma_load_2d_pair(sb + SP::kBBytes, &bmap_lo, fb, k * kBK, brow);
              }
            } else {
              if (need_b) mbar_expect_tx(fb, SP::kStageBytes);
              tma_load_4d(sa, am, fb, e.y, x0 + e.w, y0 + e.z, img);
              if (SPLIT) tma_load_4d(sa + SP::kABytes, am + 1, fb, e.y, x0 + e.w, y0 + e.z, img);
              if (need_b) {
                tma_load_2d(sb, &bmap_hi, fb, k * kBK, brow);
                if (SPLIT) tma_load_2d(sb + SP::kBBytes, &bmap_lo, fb, k * kBK, brow);
              }
            }
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 && leader) {
    // =============================== MMA issuer (pairs: leader CTA only) ========
    {
      constexpr uint32_t idesc = make_idesc(BN, kBM * CG);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t cc = 0;                                   // chunk counter (persists across tiles)
      uint32_t hcount = 0;                               // HALO: halo tiles consumed
      long long t_wait_tempty = 0, t_wait_full = 0, t_first_full = 0;
      const long long t_start = clock64();
      const int G = p.chunk_kb;
      const int S = p.split_k;
      for (int w = blockIdx.x / CG; w < p.total_tiles * S; w += gridDim.x / CG) {
        const int ks = w % S;
        const int kbeg = (ks * p.nkb) / S, kend = ((ks + 1) * p.nkb) / S;
        for (int k0 = kbeg; k0 < kend; k0 += G, ++cc) {
          const uint32_t buf = cc % NBUF;
          const uint32_t bphase = (cc / NBUF) & 1;
          const long long tA = (IDC_CTA_COUNTERS && p.dbgbuf) ? clock64() : 0;
          mbar_wait(smem_u32(&tempty_bar[buf]), bphase ^ 1, p.err, 2);
          if (IDC_CTA_COUNTERS && p.dbgbuf) t_wait_tempty += clock64() - tA;
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + buf * SP::kBufCols;
          const int k1 = (k0 + G < kend) ? k0 + G : kend;
          for (int k = k0; k < k1; ++k) {
            const long long tB = (IDC_CTA_COUNTERS && p.dbgbuf) ? clock64() : 0;
            uint32_t hslot = 0;
            if (HALO) {
              if (k % 9 == 0) {
                mbar_wait(smem_u32(&afull_bar[hcount & 1]), (hcount >> 1) & 1, p.err, 7);
                ++hcount;
              }
              hslot = (hcount - 1) & 1;
            }
            mbar_wait(smem_u32(&full_bar[stage]), phase, p.err, 3);
            if (IDC_CTA_COUNTERS && p.dbgbuf) {
              t_wait_full += clock64() - tB;
              if (t_first_full == 0) t_first_full = clock64() - t_kernel0;
            }
            tc_fence_after();
            if (elect_one()) {
            const uint32_t sa = smem_u32(smem + stage * SP::kStageBytes);
            const uint32_t sb = sa + (SPLIT ? 2 : 1) * SP::kAStage;
            const uint64_t b_hi = make_sw128_desc(sb);
            const uint64_t b_lo = make_sw128_desc(sb + SP::kBBytes);
            const uint32_t fresh = (k == k0) ? 0u : 1u;    // first MMA into a chunk buffer overwrites it
            uint32_t ha = 0;                               // HALO: this tap's window inside the halo slot
            if (HALO) {
              const int4 e = __ldg(p.kblk + k);
              ha = smem_u32(s_halo + hslot * SP::kHaloSlot) + (uint32_t)(e.z * kHaloW + e.w) * 128u;
            }
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
              const uint64_t a_hi = HALO ? make_sw128_desc(ha, kHaloW * 128) : make_sw128_desc(sa + mt * (kBM * kBK * 2));
              const uint64_t a_lo = HALO ? make_sw128_desc(ha + kHaloPlane, kHaloW * 128)
                                         : make_sw128_desc(sa + SP::kABytes + mt * (kBM * kBK * 2));
              const uint32_t d = d_tmem + mt * BN;
              uint32_t first = fresh;
              if (SPLIT) {
                // the 8 small cross terms first (accumulator still tiny -> their truncation is harmless),
                // then the 4 dominant hi*hi terms
#pragma unroll
                for (int kk = 0; kk < kBK / 16; ++kk) {
                  const uint64_t adv = (uint64_t)(kk * 2);  // 16 FP16 = 32 bytes = 2 descriptor units
                  if (PAIR) {
                    umma_f16_pair(d, a_lo + adv, b_hi + adv, idesc, first);
                    umma_f16_pair(d, a_hi + adv, b_lo + adv, idesc, 1u);
                  } else {
                    umma_f16(d, a_lo + adv, b_hi + adv, idesc, first);
                    umma_f16(d, a_hi + adv, b_lo + adv, idesc, 1u);
                  }
                  first = 1u;
                }
              }
#pragma unroll
              for (int kk = 0; kk < kBK / 16; ++kk) {
                const uint64_t adv = (uint64_t)(kk * 2);
                if (PAIR) umma_f16_pair(d, a_hi + adv, b_hi + adv, idesc, first);
                else umma_f16(d, a_hi + adv, b_hi + adv, idesc, first);
                first = 1u;
              }
            }
            if (PAIR) {
              umma_commit_pair(smem_u32(&empty_bar[stage]));                       // both CTAs' stages
              if (HALO && k % 9 == 8) umma_commit_pair(smem_u32(&aempty_bar[hslot]));   // both CTAs' halo slots
              if (k == k1 - 1) umma_commit_pair(smem_u32(&tfull_bar[buf]));        // both CTAs' accumulate warps
            } else {
              umma_commit(smem_u32(&empty_bar[stage]));   // frees the smem stage when these MMAs retire
              if (HALO && k % 9 == 8) umma_commit(smem_u32(&aempty_bar[hslot]));
              if (k == k1 - 1) umma_commit(smem_u32(&tfull_bar[buf]));   // chunk complete -> accumulate warps
            }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
      if (IDC_CTA_COUNTERS && p.dbgbuf && lane == 0) {
        p.dbgbuf[blockIdx.x * 16 + 0] = clock64() - t_start;
        p.dbgbuf[blockIdx.x * 16 + 1] = t_wait_tempty;
        p.dbgbuf[blockIdx.x * 16 + 2] = t_wait_full;
        p.dbgbuf[blockIdx.x * 16 + 6] = t_first_full;          // kernel entry -> first operand stage landed
        p.dbgbuf[blockIdx.x * 16 + 10] = t_start - t_kernel0;  // kernel entry -> MMA role entered (prologue)
      }
    }
  } else if (warp >= 4) {
    // ====================== accumulate + epilogue (8 warps) ======================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kAccRegs));
    constexpr int CH = SP::kCH;              // accumulator columns per thread
    const int quarter = warp & 3;            // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;        // MT==1: column half of the tile; MT==2: which M-tile
    const int row = quarter * 32 + lane;     // pixel row of the tile
    const int et = threadIdx.x - 128;        // 0..255
    const int c_base = (MT == 2) ? 0 : half * CH;          // first output column of this thread
    const int t_base = (MT == 2) ? half * BN : half * CH;   // its first TMEM column inside a chunk buffer
    uint32_t cc = 0;
    long long t_epi = 0, t_wait_tfull = 0, t_drain = 0, t_splitk = 0, t_spin = 0;
    const int tiles_per_img = p.tiles_y * p.tiles_x;
    const int G = p.chunk_kb;
    const int S = p.split_k;
    int staged_key = -1;
    for (int w = blockIdx.x / CG; w < p.total_tiles * S; w += gridDim.x / CG) {
      const int tile = w / S, ks = w - tile * S;
      const int kbeg = (ks * p.nkb) / S, kend = ((ks + 1) * p.nkb) / S;
      int r = tile;
      const int nt = r % p.n_tiles_n;
      r /= p.n_tiles_n;
      const int cls = r % p.ncls;
      r /= p.ncls;
      if (PAIR) r = 2 * r + (int)cta_rank;
      const int img_rel = r / tiles_per_img;
      r -= img_rel * tiles_per_img;
      const int img = p.img0 + img_rel;
      const int r2 = r;
      const int y = (r / p.tiles_x) * (p.hbox * MT) + (MT == 2 ? half * p.hbox : 0) + (row >> p.wshift);
      const int x = (r % p.tiles_x) * p.wbox + (row & (p.wbox - 1));
      const bool valid = y < p.Hl && x < p.Wl && img < p.n_img;   // pairs: an odd tile count leaves one dummy tile
      const int n0 = nt * BN;
      // stage this tile's per-channel epilogue vectors -- only when they change (n-tile, or image when a
      // global-hints vector is added); for the single-n-tile layers that is once per kernel
      const int vkey = p.gadd ? (img * p.n_tiles_n + nt) : nt;
      if (vkey != staged_key) {
        asm volatile("bar.sync 1, 256;" ::: "memory");      // previous tile's readers are done
        for (int i = et; i < BN; i += kAccThreads) {
          s_bias[i] = p.bias[n0 + i];
          s_scale[i] = p.scale[n0 + i];
          // pairs: the dummy tile of an odd tile count has img == n_img -> clamp (its rows are never stored)
          const int gi = img < p.n_img ? img : p.n_img - 1;
          s_shift[i] = p.shift[n0 + i] + (p.gadd ? p.gadd[(size_t)gi * p.gadd_ld + n0 + i] * p.gadd_mult : 0.f);
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        staged_key = vkey;
      }

      float acc[CH];
#pragma unroll
      for (int j = 0; j < CH; ++j) acc[j] = 0.f;
      for (int k0 = kbeg; k0 < kend; k0 += G, ++cc) {
        const uint32_t buf = cc % NBUF;
        const uint32_t bphase = (cc / NBUF) & 1;
        const long long tC = (IDC_CTA_COUNTERS && p.dbgbuf) ? clock64() : 0;
        mbar_wait(smem_u32(&tfull_bar[buf]), bphase, p.err, 4);
        const long long tD = (IDC_CTA_COUNTERS && p.dbgbuf) ? clock64() : 0;
        t_wait_tfull += tD - tC;
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * SP::kBufCols + t_base;
        if (CH >= 128) {     // 64 columns in flight per TMEM round trip (232-register budget after setmaxnreg)
#pragma unroll
          for (int pc = 0; pc < CH / 64; ++pc) {
            uint32_t v0[32], v1[32];
            tmem_ld32(taddr + pc * 64, v0);
            tmem_ld32(taddr + pc * 64 + 32, v1);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[pc * 64 + j] += __uint_as_float(v0[j]);   // FP32 round-to-nearest
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[pc * 64 + 32 + j] += __uint_as_float(v1[j]);
          }
        } else if (CH == 64) {   // both loads in flight before the wait: hides one TMEM round trip per chunk
          uint32_t v0[32], v1[32];
          tmem_ld32(taddr, v0);
          tmem_ld32(taddr + 32, v1);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[j] += __uint_as_float(v0[j]);
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[(32 + j) % CH] += __uint_as_float(v1[j]);
        } else {
#pragma unroll
          for (int pc = 0; pc < CH / 32; ++pc) {
            uint32_t v[32];
            tmem_ld32(taddr + pc * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[pc * 32 + j] += __uint_as_float(v[j]);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR && !leader) mbar_arrive_rank0(smem_u32(&tempty_bar[buf]));   // the leader's MMA warp owns the buffers
          else mbar_arrive(smem_u32(&tempty_bar[buf]));
        }
        if (IDC_CTA_COUNTERS && p.dbgbuf) t_drain += clock64() - tD;
      }
      const long long tE = (IDC_CTA_COUNTERS && p.dbgbuf) ? clock64() : 0;

      // ---- split-K: park the partial tile in the workspace, wait until all S slices of this tile have
      //      arrived (they are co-resident: work items <= #SMs by construction), then every CTA reduces and
      //      finishes ITS share of the 16-column pieces (piece % S == ks), summing the slices in fixed order
      //      (deterministic).  Arrive/depart counters reset themselves for the next launch / graph replay. ----
      if (S > 1) {
        // workspace layout [work item][column quad][row] (float4): lanes = rows -> 512-byte coalesced
        // pairs: each CTA of the pair parks / reduces its own 128 rows (slot = work item * CG + rank)
        float4* wp = reinterpret_cast<float4*>(p.ws) + ((size_t)(w * CG + (int)cta_rank) * (MT * BN / 4) + t_base / 4) * kBM + row;
        // kSkipOwn (<= 64 accumulators per thread, i.e. the 128-column tiles): the pieces this CTA finishes itself stay
        // in registers -- 1/S of the park traffic and one slice of the reduction reads less
        constexpr bool kSkipOwn = CH <= 64;
#pragma unroll
        for (int j = 0; j < CH; j += 4) {
          if (kSkipOwn && ((c_base + j) >> 5) % S == ks) continue;
          __stcg(wp + (size_t)(j / 4) * kBM, make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]));
        }
        __threadfence();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (et == 0) {
          int* cnt = p.counters + 2 * (tile * CG + (int)cta_rank);
          atomicAdd(cnt, 1);
          const long long t0 = clock64();
          int seen;
          do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(cnt) : "memory");
            if (seen < S && clock64() - t0 > 6000000000LL) mbar_timeout(p.err, 5);
          } while (seen < S);
          if (IDC_CTA_COUNTERS && p.dbgbuf) t_spin += clock64() - t0;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
#pragma unroll
        for (int ch = 0; ch < CH; ch += 32) {
          if (((c_base + ch) >> 5) % S != ks) continue;
          // kSkipOwn: the accumulator already holds this CTA's own slice; the other slices are added to it in slice
          // order (the order is a function of (piece, S) only, so results stay deterministic)
          if (!kSkipOwn) {
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[ch + j] = 0.f;
          }
          // The slices are summed in slice order (deterministic, same order as a serial loop), but the loads of QB
          // slices are issued together: a serial loop pays one L2 round trip (~700 cycles) per slice -- measured
          // 9 of the 10.3 kcycles this section took per launch at batch 1 (profiles/r02_cta_counters_batch1.txt).
          constexpr int QB = kSkipOwn ? 3 : ((CH >= 128) ? 2 : 4);   // register budget: CH accumulators + QB * 32 in flight
          const float4* rp0 = reinterpret_cast<const float4*>(p.ws) +
                              ((size_t)(tile * S * CG + (int)cta_rank) * (MT * BN / 4) + (t_base + ch) / 4) * kBM + row;
          const size_t qstride = (size_t)CG * (MT * BN / 4) * kBM;
          const int n_other = kSkipOwn ? S - 1 : S;        // slices to fetch (kSkipOwn: all but this CTA's own)
          for (int i0 = 0; i0 < n_other; i0 += QB) {
            float4 v[QB][8];
#pragma unroll
            for (int qq = 0; qq < QB; ++qq) {
              const int i = (i0 + qq < n_other) ? i0 + qq : i0;      // tail: re-read a valid slice, discarded below
              const int q = kSkipOwn ? i + (i >= ks ? 1 : 0) : i;
#pragma unroll
              for (int j = 0; j < 8; ++j) v[qq][j] = __ldcg(rp0 + (size_t)q * qstride + (size_t)j * kBM);
            }
#pragma unroll
            for (int qq = 0; qq < QB; ++qq) {
              if (i0 + qq < n_other) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  acc[ch + 4 * j] += v[qq][j].x; acc[ch + 4 * j + 1] += v[qq][j].y;
                  acc[ch + 4 * j + 2] += v[qq][j].z; acc[ch + 4 * j + 3] += v[qq][j].w;
                }
              }
            }
          }
        }
      }
      if (IDC_CTA_COUNTERS && p.dbgbuf && S > 1) t_splitk += clock64() - tE;
      // ---- epilogue on the register accumulators, 32 output channels at a time.  The output kind is uniform for
      //      the launch, so the branch sits outside the slab loops; the per-channel vectors are read with
      //      ld.shared (warp-uniform 16-byte reads), never through generic addressing. ----
      const uint32_t sv = epi_token(smem_u32(s_bias) + (uint32_t)c_base * 4u);   // bias | +BN*4: scale | +2*BN*4: shift
      const float neg_slope = p.act == ACT_RELU ? 0.f : (p.act == ACT_LEAKY02 ? 0.2f : 1.f);
      auto slab = [&](const int ch, float (&f)[32]) {
#pragma unroll
        for (int j4 = 0; j4 < 32; j4 += 4) {
          const float4 vb = ld_shared_f4(sv + (uint32_t)(ch + j4) * 4u);
          const float4 vs = ld_shared_f4(sv + (uint32_t)(BN + ch + j4) * 4u);
          const float4 vt = ld_shared_f4(sv + (uint32_t)(2 * BN + ch + j4) * 4u);
          const float b4[4] = {vb.x, vb.y, vb.z, vb.w}, s4[4] = {vs.x, vs.y, vs.z, vs.w}, t4[4] = {vt.x, vt.y, vt.z, vt.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            // one branch-free form for none / ReLU / LeakyReLU(0.2): max(t, slope*t) with slope = 1 / 0 / 0.2
            // (slope <= 1, so slope*t >= t exactly when t <= 0; one rounding, same value as slope*t alone)
            const float t = acc[ch + j4 + j] + b4[j];
            const float a = fmaxf(t, neg_slope * t);
            f[j4 + j] = fmaf(a, s4[j], t4[j]);
          }
        }
      };
      if (p.wout) {
        // fused model_out: conv1x1(128->2) + tanh, x110 (model.py:108-109,175)
        const uint32_t sh = epi_token(smem_u32(s_head) + (uint32_t)c_base * 4u);
        float h0 = 0.f, h1 = 0.f;
#pragma unroll
        for (int ch = 0; ch < CH; ch += 32) {
          float f[32];
          slab(ch, f);
#pragma unroll
          for (int j4 = 0; j4 < 32; j4 += 4) {
            const float4 w0 = ld_shared_f4(sh + (uint32_t)(ch + j4) * 4u);
            const float4 w1 = ld_shared_f4(sh + (uint32_t)(128 + ch + j4) * 4u);
            h0 = fmaf(f[j4], w0.x, fmaf(f[j4 + 1], w0.y, fmaf(f[j4 + 2], w0.z, fmaf(f[j4 + 3], w0.w, h0))));
            h1 = fmaf(f[j4], w1.x, fmaf(f[j4 + 1], w1.y, fmaf(f[j4 + 2], w1.z, fmaf(f[j4 + 3], w1.w, h1))));
          }
        }
        // the two column halves of a pixel live in two warps when MT == 1 -> combine through smem
        if (MT == 1) {
          if (half == 1) { s_red[row * 2] = h0; s_red[row * 2 + 1] = h1; }
          asm volatile("bar.sync 2, 256;" ::: "memory");
          if (half == 0) { h0 += s_red[row * 2]; h1 += s_red[row * 2 + 1]; }
          asm volatile("bar.sync 2, 256;" ::: "memory");     // s_red is rewritten by the next tile
        }
        if ((MT == 2 || half == 0) && valid) {
          const size_t HW = (size_t)p.Hl * p.Wl;
          const size_t o = (size_t)img * 2 * HW + (size_t)y * p.Wl + x;
          p.out_ab[o] = tanhf(h0 + s_head[256]) * p.out_mult;           // out_mult = 110 (model.py:175) or 100 (Caffe spec)
          p.out_ab[o + HW] = tanhf(h1 + s_head[257]) * p.out_mult;
        }
      } else if (p.out_f32) {
        float* o32 = p.out_f32 + ((size_t)(img * p.Hl + y) * p.Wl + x) * p.out_ld + n0 + c_base;
#pragma unroll
        for (int ch = 0; ch < CH; ch += 32) {
          if (S > 1 && ((c_base + ch) >> 5) % S != ks) continue;   // another CTA of the split finishes this piece
          float f[32];
          slab(ch, f);
          if (valid) {
            float4* o = reinterpret_cast<float4*>(o32 + ch);
#pragma unroll
            for (int q = 0; q < 8; ++q) o[q] = make_float4(f[4 * q], f[4 * q + 1], f[4 * q + 2], f[4 * q + 3]);
          }
        }
      } else {
        // activation store, warp-transposed: the warp's 32 rows x 64 bytes go through a private 2 KB smem tile
        // (XOR-swizzled, conflict-free both ways) so that each store instruction writes 8 pixel rows x 64
        // contiguous bytes instead of 32 rows x 16 bytes -- 4x fewer L1 transactions.  Store instruction i of a
        // slab covers rows i*8 + lane/4 of this warp's 32 rows; rows outside the image get a null pointer.
        const int ty0 = (r2 / p.tiles_x) * (p.hbox * MT) + (MT == 2 ? half * p.hbox : 0);
        const int tx0 = (r2 % p.tiles_x) * p.wbox;
        __half* ph[4];
        const ptrdiff_t lo_delta = SPLIT ? p.out_lo - p.out_hi : 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int rr = quarter * 32 + i * 8 + (lane >> 2);
          const int yy = ty0 + (rr >> p.wshift), xx = tx0 + (rr & (p.wbox - 1));
          const bool ok = yy < p.Hl && xx < p.Wl && img < p.n_img;
          ph[i] = ok ? p.out_hi + ((size_t)(img * p.Hout + yy * p.os + (cls >> 1)) * p.Wout + xx * p.os + (cls & 1)) * p.Cout +
                           n0 + c_base + (lane & 3) * 8
                     : nullptr;
        }
        const uint32_t wbuf = smem_u32(s_out) + (warp - 4) * 2048;
        const uint32_t wst = wbuf + lane * 64, wsw = (lane >> 1) & 3;
        uint32_t wld[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int rl = i * 8 + (lane >> 2), c = lane & 3;          // row of this warp's 32, 16-byte chunk
          wld[i] = wbuf + rl * 64 + ((c ^ ((rl >> 1) & 3)) << 4);
        }
#pragma unroll
        for (int ch = 0; ch < CH; ch += 32) {
          if (S > 1 && ((c_base + ch) >> 5) % S != ks) continue;
          float f[32];
          slab(ch, f);
          uint32_t hw[16], lw[16];
          split_pack<SPLIT>(f, hw, lw);
#pragma unroll
          for (int plane = 0; plane < (SPLIT ? 2 : 1); ++plane) {
            const uint32_t* src = plane == 0 ? hw : lw;
#pragma unroll
            for (int c = 0; c < 4; ++c)
              st_shared_v4(wst + ((c ^ wsw) << 4), make_uint4(src[4 * c], src[4 * c + 1], src[4 * c + 2], src[4 * c + 3]));
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              uint4 v;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                           : "r"(wld[i]));
              if (ph[i]) *reinterpret_cast<uint4*>(ph[i] + (plane ? lo_delta : 0) + ch) = v;
            }
            __syncwarp();
          }
        }
      }
      if (IDC_CTA_COUNTERS && p.dbgbuf) t_epi += clock64() - tE;
      if (S > 1) {
        asm volatile("bar.sync 1, 256;" ::: "memory");          // all of this CTA's workspace reads are done
        if (et == 0) {
          int* cnt = p.counters + 2 * (tile * CG + (int)cta_rank);
          if (atomicAdd(cnt + 1, 1) == S - 1) { cnt[0] = 0; cnt[1] = 0; __threadfence(); }
        }
      }
    }
    t_wait_tfull_g = t_wait_tfull; t_drain_g = t_drain; t_epi_g = t_epi; t_splitk_g = t_splitk; t_spin_g = t_spin;
  }

  // ---- teardown ----
  if (IDC_CTA_COUNTERS && p.dbgbuf && warp == 4 && lane == 0) {
    p.dbgbuf[blockIdx.x * 16 + 3] = t_wait_tfull_g;
    p.dbgbuf[blockIdx.x * 16 + 4] = t_drain_g;
    p.dbgbuf[blockIdx.x * 16 + 5] = t_epi_g;
    p.dbgbuf[blockIdx.x * 16 + 7] = clock64() - t_kernel0;     // CTA lifetime up to the teardown
    p.dbgbuf[blockIdx.x * 16 + 8] = t_splitk_g;                // split-K: park + wait + reduce
    p.dbgbuf[blockIdx.x * 16 + 9] = t_spin_g;                  // split-K: of which spinning for the other slices
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();   // pairs: the peer may still arrive on / read from this CTA
  if (warp == 1) {
    __syncwarp();
    if (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)SP::kTmemCols)
                   : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)SP::kTmemCols)
                   : "memory");
  }
}

template <int BN, int MT, int CG, bool SPLIT, bool HALO = false>
__global__ void __launch_bounds__(kThreads, 1)
umma_conv_kernel(const __grid_constant__ CUtensorMap bmap_hi, const __grid_constant__ CUtensorMap bmap_lo,
                 const __grid_constant__ UmmaParams p) {
  conv_body<BN, MT, CG, SPLIT, HALO>(bmap_hi, bmap_lo, p);
}

// ------------------------------------------------------------------------------------------
// conv1_1 on the tensor cores: the input pack cat(L/100, ab/110, mask - maskcent) (model.py:142-148) + model1.0
// (4 -> 64, 3x3, ReLU; model.py:13-14) as ONE padded k-block.  K = 9 taps x 4 channels = 36 -> 48 (three K=16 steps).
// There is no 16-byte granule to aim a TMA box at (a tap contributes 4 channels = 8 bytes), so the 128 threads of a CTA
// gather and normalise their pixel's 36 inputs themselves, split them into FP16 hi / lo (x 2^6, like every activation)
// and write their row of the two K-major SWIZZLE_128B operand tiles directly; the 64 x 48 weight tile (hi / lo,
// pre-swizzled by conv1_1_pack_kernel) stays in shared memory for the life of the CTA.  9 MMAs (lo*hi, hi*lo, hi*hi per
// K step) replace 2304 FFMAs per pixel; the epilogue (bias, ReLU, hi/lo split, warp-transposed stores) is the FP32
// kernel's.  4 CTAs per SM hide each other's gather / MMA / epilogue phases (no intra-CTA pipeline).
// ------------------------------------------------------------------------------------------
constexpr int kC11K = 48;                       // padded K (3 MMA steps of 16)
constexpr int kC11PackBytes = 2 * 8192 + 2 * 64 * 4;   // [B hi | B lo] smem images + bias' + scale'
constexpr int kC11Smem = 2 * 16384 + kC11PackBytes + 64 + 1024;   // A hi/lo, pack, barrier + tmem ptr, alignment slack

__device__ __forceinline__ uint32_t sw128_off(int row, int chunk) {   // byte offset of a 16-byte chunk in a K-major SW128 tile
  return (uint32_t)((row >> 3) * 1024 + (row & 7) * 128 + ((chunk ^ (row & 7)) << 4));
}

// one thread per output channel: power-of-two scale so the largest weight lands in [256, 512), hi/lo split, swizzled
// smem image of the [64 cout][48 k] tile (k = tap * 4 + cin, zero beyond 36), bias' = bias * 2^6 * 2^e, scale' = 2^-e
__global__ void conv1_1_pack_kernel(const float* __restrict__ w36x64, const float* __restrict__ bias, uint8_t* __restrict__ out) {
  const int co = threadIdx.x;
  if (co >= 64) return;
  float mx = 0.f;
  for (int k = 0; k < 36; ++k) mx = fmaxf(mx, fabsf(w36x64[k * 64 + co]));
  int e = 0;
  if (mx > 0.f) { int ex; frexpf(mx, &ex); e = 9 - ex; }        // mx * 2^e in [256, 512)
  const float sc = ldexpf(1.f, e);
  __half* bh = reinterpret_cast<__half*>(out);
  __half* bl = reinterpret_cast<__half*>(out + 8192);
  for (int k = 0; k < 64; ++k) {
    const float v = k < 36 ? w36x64[k * 64 + co] * sc : 0.f;
    __half hi, lo;
    split_h(v, hi, lo);
    const uint32_t o = (sw128_off(co, k >> 3) >> 1) + (k & 7);
    bh[o] = hi; bl[o] = lo;
  }
  float* vec = reinterpret_cast<float*>(out + 16384);
  vec[co] = bias[co] * kActScale * sc;
  vec[64 + co] = ldexpf(1.f, -e);
}

template <bool SPLIT>
__global__ void __launch_bounds__(128, 4)
conv1_1_umma_kernel(const uint8_t* __restrict__ pack, const float* __restrict__ L, const float* __restrict__ ab,
                    const float* __restrict__ mask, float maskcent, int N, int H, int Wd, __half* __restrict__ ohi,
                    __half* __restrict__ olo, int* err) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_ahi = smem;                       // [128 px][64 k] FP16, K-major SW128 (16 KB); reused as the store staging
  uint8_t* s_alo = smem + 16384;
  uint8_t* s_pack = smem + 32768;              // B hi (8 KB) | B lo (8 KB) | bias' | scale'
  const float* s_vec = reinterpret_cast<const float*>(s_pack + 16384);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_pack + kC11PackBytes);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // ---- setup: barrier, 64 TMEM columns, the packed weight tile ----
  if (threadIdx.x == 0) {
    mbar_init(smem_u32(s_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(64u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  {
    const uint4* src = reinterpret_cast<const uint4*>(pack);
    uint4* dst = reinterpret_cast<uint4*>(s_pack);
    for (int i = threadIdx.x; i < kC11PackBytes / 16; i += 128) dst[i] = __ldg(src + i);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // the weight tile is read by the tensor core (async proxy)
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;
  pdl_launch_dependents();
  pdl_wait();

  const size_t HW = (size_t)H * Wd, total = (size_t)N * HW;
  const int ntiles = (int)((total + 127) / 128);
  constexpr uint32_t idesc = make_idesc(64, kBM);
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const size_t pix = (size_t)tile * 128 + threadIdx.x;
    const bool live = pix < total;
    const size_t pixc = live ? pix : 0;
    const int n = (int)(pixc / HW);
    const int r = (int)(pixc - (size_t)n * HW);
    const int y = r / Wd, x = r - y * Wd;
    // ---- gather + normalise + split: this thread's row of the A tiles (k = tap * 4 + channel) ----
    float in[kC11K];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int iy = y + ky - 1, ix = x + kx - 1;
        const bool ok = live && iy >= 0 && iy < H && ix >= 0 && ix < Wd;
        const size_t o = (size_t)iy * Wd + ix;
        const int t = (ky * 3 + kx) * 4;
        // zero padding applies to the concatenated, normalised input (model.py:148 then Conv2d pad)
        const float l = ok ? __ldg(L + (size_t)n * HW + o) : 0.f;
        const float a = ok ? __ldg(ab + (size_t)n * 2 * HW + o) : 0.f;
        const float b = ok ? __ldg(ab + (size_t)n * 2 * HW + HW + o) : 0.f;
        const float m = ok ? __ldg(mask + (size_t)n * HW + o) - maskcent : 0.f;
        const float ql = l * 0.01f, qa = a * (1.0f / 110.0f), qb = b * (1.0f / 110.0f);
        in[t + 0] = fmaf(fmaf(-ql, 100.0f, l), 0.01f, ql);                    // x / 100, correctly rounded (cf. div_corrected)
        in[t + 1] = fmaf(fmaf(-qa, 110.0f, a), 1.0f / 110.0f, qa);
        in[t + 2] = fmaf(fmaf(-qb, 110.0f, b), 1.0f / 110.0f, qb);
        in[t + 3] = m;
      }
#pragma unroll
    for (int k = 36; k < kC11K; ++k) in[k] = 0.f;
#pragma unroll
    for (int j = 0; j < kC11K / 8; ++j) {
      uint32_t hw[4], lw[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float v0 = in[8 * j + 2 * q] * kActScale, v1 = in[8 * j + 2 * q + 1] * kActScale;
        hw[q] = pack_f16x2_sat(v0, v1);
        const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hw[q]));
        lw[q] = pack_f16x2_sat(v0 - hf.x, v1 - hf.y);
      }
      const uint32_t o = sw128_off(threadIdx.x, j);
      st_shared_v4(smem_u32(s_ahi) + o, make_uint4(hw[0], hw[1], hw[2], hw[3]));
      if (SPLIT) st_shared_v4(smem_u32(s_alo) + o, make_uint4(lw[0], lw[1], lw[2], lw[3]));
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core reads
    __syncthreads();
    // ---- 9 MMAs into 64 TMEM columns: the small cross terms first, then hi*hi (as in umma_conv_kernel) ----
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        const uint64_t a_hi = make_sw128_desc(smem_u32(s_ahi)), a_lo = make_sw128_desc(smem_u32(s_alo));
        const uint64_t b_hi = make_sw128_desc(smem_u32(s_pack)), b_lo = make_sw128_desc(smem_u32(s_pack) + 8192);
        uint32_t first = 0u;
        if (SPLIT) {
#pragma unroll
          for (int kk = 0; kk < kC11K / 16; ++kk) {
            const uint64_t adv = (uint64_t)(kk * 2);
            umma_f16(tmem, a_lo + adv, b_hi + adv, idesc, first);
            umma_f16(tmem, a_hi + adv, b_lo + adv, idesc, 1u);
            first = 1u;
          }
        }
#pragma unroll
        for (int kk = 0; kk < kC11K / 16; ++kk) {
          const uint64_t adv = (uint64_t)(kk * 2);
          umma_f16(tmem, a_hi + adv, b_hi + adv, idesc, first);
          first = 1u;
        }
        umma_commit(smem_u32(s_bar));
      }
      __syncwarp();
    }
    mbar_wait(smem_u32(s_bar), phase, err, 9);
    phase ^= 1;
    tc_fence_after();
    // ---- epilogue: row = pixel; relu(acc + bias') * scale' = 2^6 * relu(conv + b) -> hi / lo -> coalesced stores ----
    uint32_t v0[32], v1[32];
    const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16);
    tmem_ld32(taddr, v0);
    tmem_ld32(taddr + 32, v1);
    tmem_ld_wait();
    tc_fence_before();
    float f[64];
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      f[c] = fmaxf(__uint_as_float(v0[c]) + s_vec[c], 0.f) * s_vec[64 + c];
      f[32 + c] = fmaxf(__uint_as_float(v1[c]) + s_vec[32 + c], 0.f) * s_vec[96 + c];
    }
    // the operand tiles are consumed (the commit has arrived): reuse their memory as the per-warp transpose tiles
    uint4* tilew = reinterpret_cast<uint4*>(s_ahi) + warp * 256;     // 32 rows x 8 chunks of 16 B = 4 KB per warp
    const size_t wpix0 = (size_t)tile * 128 + warp * 32;
#pragma unroll
    for (int plane = 0; plane < (SPLIT ? 2 : 1); ++plane) {
#pragma unroll
      for (int c8 = 0; c8 < 8; ++c8) {
        uint32_t w4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float a0 = f[c8 * 8 + 2 * q], a1 = f[c8 * 8 + 2 * q + 1];
          const uint32_t hw = pack_f16x2_sat(a0, a1);
          if (plane == 0) {
            w4[q] = hw;
          } else {
            const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hw));
            w4[q] = pack_f16x2_sat(a0 - hf.x, a1 - hf.y);
          }
        }
        tilew[lane * 8 + (c8 ^ (lane & 7))] = make_uint4(w4[0], w4[1], w4[2], w4[3]);
      }
      __syncwarp();
      __half* gbase = (plane == 0 ? ohi : olo) + wpix0 * 64;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rl = i * 4 + (lane >> 3), c = lane & 7;
        if (wpix0 + rl < total) reinterpret_cast<uint4*>(gbase)[i * 32 + lane] = tilew[rl * 8 + (c ^ (rl & 7))];
      }
      __syncwarp();
    }
    __syncthreads();        // TMEM drained and staging read by every warp before the next tile overwrites either
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(64u) : "memory");
}

cudaError_t conv1_1_umma_pack(Ctx* c) {
  if (!c->w11_umma) {
    cudaError_t e = cudaMalloc(&c->w11_umma, kC11PackBytes);
    if (e != cudaSuccess) return e;
  }
  conv1_1_pack_kernel<<<1, 64>>>(c->w11, c->b11, c->w11_umma);
  cudaError_t e = cudaGetLastError();
  return e != cudaSuccess ? e : cudaDeviceSynchronize();
}

cudaError_t launch_conv1_1_umma(Ctx* c, int n, const float* L, const float* ab, const float* mask, float maskcent,
                                cudaStream_t st, int img0) {
  const ActBuf& o = c->bufs[c->buf_index.at("a1_1")];
  const size_t HW = (size_t)o.H * o.W, npix = (size_t)n * HW, ooff = (size_t)img0 * HW * o.C;
  const int ntiles = (int)((npix + 127) / 128);
  static int sms[64] = {};
  int& nsm = sms[c->dev < 64 ? c->dev : 0];
  if (!nsm) { cudaDeviceProp prop; cudaGetDeviceProperties(&prop, c->dev); nsm = prop.multiProcessorCount; }
  const int grid = ntiles < 4 * nsm ? ntiles : 4 * nsm;
  L += img0 * HW; ab += img0 * 2 * HW; mask += img0 * HW;
  static unsigned long long attr_devs = 0;
  if (c->dev >= 64 || !(attr_devs & (1ull << c->dev))) {
    cudaError_t e = cudaFuncSetAttribute(conv1_1_umma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kC11Smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv1_1_umma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kC11Smem);
    if (e != cudaSuccess) return e;
    if (c->dev < 64) attr_devs |= 1ull << c->dev;
  }
  __half* hi = static_cast<__half*>(o.p0) + ooff;
  __half* lo = o.p1 ? static_cast<__half*>(o.p1) + ooff : nullptr;
  cudaError_t e = lo ? launch_k(c, conv1_1_umma_kernel<true>, dim3(grid), dim3(128), (size_t)kC11Smem, st, c->w11_umma, L, ab, mask,
                                maskcent, n, o.H, o.W, hi, lo, c->d_err)
                     : launch_k(c, conv1_1_umma_kernel<false>, dim3(grid), dim3(128), (size_t)kC11Smem, st, c->w11_umma, L, ab, mask,
                                maskcent, n, o.H, o.W, hi, lo, c->d_err);
  c->launch_count++;
  return e;
}

// ------------------------------------------------------------------------------------------
// host side: tensor maps + launch plan
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

struct UmmaPlan {
  CUtensorMap* d_amaps = nullptr;
  int4* d_kblk = nullptr;
  CUtensorMap bmap_hi, bmap_lo;
  UmmaParams prm{};
  int num_sms = 148;
  int dev = 0;
  int mt = 1;               // M-tiles (128 pixels each) per CTA tile
  int cg = 1;               // 2: CTA pairs (cta_group::2), one 256x256 output tile per pair
  int split_k = 1;
  bool halo = false;        // one halo tile per input-channel group instead of one TMA box per tap (stride-1 3x3 layers)
  size_t ws_floats = 0;
  int ws_tiles = 0;
};

struct ViewKey {
  int src, s, qy, qx;
  bool operator==(const ViewKey& o) const { return src == o.src && s == o.s && qy == o.qy && qx == o.qx; }
};

static int floordiv2(int v) { return v >= 0 ? v / 2 : -((-v + 1) / 2); }

template <int BN, int MT, int CG, bool SPLIT, bool HALO = false>
static cudaError_t launch_inst(const UmmaPlan& pl, const UmmaParams& prm, cudaStream_t st, bool pdl) {
  using SP = SmemPlan<BN, MT, CG, SPLIT, HALO>;
  static unsigned long long attr_devs = 0;       // the opt-in is per device: one bit per device ordinal
  if (pl.dev >= 64 || !(attr_devs & (1ull << pl.dev))) {
    cudaError_t e = cudaFuncSetAttribute(umma_conv_kernel<BN, MT, CG, SPLIT, HALO>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         SP::kTotal);
    if (e != cudaSuccess) return e;
    if (pl.dev < 64) attr_devs |= 1ull << pl.dev;
  }
  const long items = (long)prm.total_tiles * prm.split_k;
  int grid = items * CG < pl.num_sms ? (int)items * CG : (pl.num_sms / CG) * CG;
  if (prm.max_ctas > 0 && grid > prm.max_ctas) grid = prm.max_ctas;   // persistent loop: any grid size covers all tiles
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = SP::kTotal;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  int na = 0;
  if (CG > 1) {
    at[na].id = cudaLaunchAttributeClusterDimension;
    at[na].val.clusterDim.x = CG; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl) {   // may start while the previous kernel of the forward drains (see pdl_wait in the kernel)
    at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = at;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, umma_conv_kernel<BN, MT, CG, SPLIT, HALO>, pl.bmap_hi, pl.bmap_lo, prm);
}

int umma_plan_op(Ctx* c, ConvOp& op) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { c->err = "cuTensorMapEncodeTiled entry point not available"; return IDC_ERR_CUDA; }
  umma_free_op(op);
  UmmaPlan* pl = new UmmaPlan();
  op.umma_plan = pl;
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, c->dev);
  pl->num_sms = prop.multiProcessorCount;
  pl->dev = c->dev;
  // tile geometry
  op.bn_tile = (op.cout_pad % 256 == 0) ? 256 : (op.cout_pad % 192 == 0) ? 192 : (op.cout_pad % 128 == 0) ? 128 : 64;
  if (op.cout_pad % op.bn_tile) { c->err = "cout not tileable: " + op.name; return IDC_ERR_ARG; }
  int best = 1 << 30;
  for (int wb = 128; wb >= 8; wb >>= 1) {
    const int hb = kBM / wb;
    const int t = ceil_div(op.Wl, wb) * ceil_div(op.Hl, hb);
    if (t < best) { best = t; op.wbox = wb; op.hbox = hb; }
  }
  // HALO: stride-1 3x3 convs of one source with 128 output columns per tile (c2_2, c9_2, c10_2: the layers that are
  // shared-memory-bandwidth bound with per-tap boxes) load one 18x10-pixel halo tile per 64 input channels instead of
  // one box per tap, when the launch fills the machine.  Measured at 64 x 256^2: c2_2 0.76 -> 0.63 ms, c9_2 0.76 ->
  // 0.63, c10_2 2.44 -> 2.28; the 64-column c1_2 gets slower (1.11 -> 1.17: its weight tile is re-streamed per 128
  // instead of 256 pixels) and keeps the per-tap path.  option halo=0 turns it off, =3 forces it on every eligible op
  // (also 64 columns, also tiny launches) for the unit tests.
  {
    const int mode = c->opt.halo;
    bool ok = mode >= 1 && !c->fast && op.ncls == 1 && op.ntaps == 9;
    unsigned seen = 0;
    for (int t = 0; ok && t < op.ntaps; ++t) {
      const Tap& tp = op.taps[0][t];
      if (tp.src != op.taps[0][0].src || op.src[tp.src].s != 1 || tp.ty < -1 || tp.ty > 1 || tp.tx < -1 || tp.tx > 1) ok = false;
      else seen |= 1u << ((tp.ty + 1) * 3 + tp.tx + 1);
    }
    if (ok && (seen != 0x1FFu || op.src[op.taps[0][0].src].cin % kBK)) ok = false;
    if (ok && !(op.bn_tile == 128 || (mode >= 3 && op.bn_tile == 64))) ok = false;
    if (ok) {   // only launches that fill the machine (the split-K path decides for itself below)
      const long T = (long)c->max_n * ceil_div(op.Hl, 16) * ceil_div(op.Wl, 8) * (op.cout_pad / op.bn_tile);
      if (T < 2L * pl->num_sms && mode < 3) ok = false;
    }
    pl->halo = ok;
    if (ok) { op.wbox = 8; op.hbox = 16; }
  }
  // Two M-tiles per CTA tile (one 256-pixel TMA box, two MMAs sharing each B tile) for the narrow-N layers:
  // halves the weight re-streaming and the per-k-block hand-off overhead.  Only when the launch still
  // fills the machine at the ctx's max batch (the batch-1 latency ctx keeps 128-pixel tiles).
  pl->mt = 1;
  if (op.bn_tile <= 128 && !pl->halo) {
    const long tiles2 = (long)op.ncls * c->max_n * ceil_div(op.Hl, 2 * op.hbox) * ceil_div(op.Wl, op.wbox) *
                        (op.cout_pad / op.bn_tile);
    if (tiles2 >= 2L * pl->num_sms && op.hbox * 2 <= 256) pl->mt = 2;
  }
  { const int v = c->opt.mt; if (!pl->halo && (v == 1 || (v == 2 && op.bn_tile <= 128))) pl->mt = v; }
  // CTA pairs for the 256-wide tiles when the launch is large (never on the split-K / batch-1 path)
  pl->cg = 1;
  {
    const long tiles1 = (long)op.ncls * c->max_n * ceil_div(op.Hl, op.hbox) * ceil_div(op.Wl, op.wbox) * (op.cout_pad / op.bn_tile);
    const bool can = !c->fast && (op.bn_tile == 256 || op.bn_tile == 128 || (op.bn_tile == 64 && (pl->mt == 2 || pl->halo)));
    const long tiles_mt = tiles1 / pl->mt;
    const int mode = c->opt.pairs;   // 0 = off, 1 (default) = launches that give every SM pair >= 2 tiles, 2 = always
    // >= 2 tiles per SM (= 4 per pair).  Measured at batch 1 (profiles/r02_latency_per_op.txt): up10 62 -> 55 us,
    // c10_2 65 -> 49 us with pairs -- these launches re-fetch their weight tile per 128-pixel tile and are bound by the
    // L2 -> SM operand traffic, which a pair halves for the weights.
    if (can && (mode >= 2 || (mode == 1 && tiles_mt >= 2L * pl->num_sms))) pl->cg = 2;
  }
  const int nkb = op.K / kBK;
  // split-K for launches that cannot fill the machine even at the ctx's max batch (interactive path): K is cut into S
  // slices per tile, all work items co-resident.  With `split_pairs` the slices run as CTA pairs (cta_group::2): per
  // k-block an SM then fetches 64 KB of operands instead of 96 KB -- at batch 1 these launches are bound by the
  // L2 -> SM operand traffic (every CTA re-fetches its A and B tiles), not by the tensor pipe.
  {
    const int ty = ceil_div(op.Hl, op.hbox * pl->mt), tx = ceil_div(op.Wl, op.wbox), ntn = op.cout_pad / op.bn_tile;
    const long m_tiles = (long)c->max_n * ty * tx;
    const long T = (long)op.ncls * m_tiles * ntn;
    int S = 1;
    const bool eligible = nkb >= 8 && !op.fuse_out_head && pl->mt == 1 && pl->cg == 1 && !pl->halo;
    if (T * 2 <= pl->num_sms && eligible) {
      S = (int)(pl->num_sms / T);
      if (S > nkb / 4) S = nkb / 4;
      if (S > op.bn_tile / 32) S = op.bn_tile / 32;      // one 32-column piece per CTA at least
      if (S < 1) S = 1;
    }
    {                                                      // experiments; must keep all work items co-resident
      const int v = c->opt.split_k;
      if (v >= 1 && v <= nkb && v <= op.bn_tile / 32 && pl->mt == 1 && !pl->halo && pl->cg == 1 && T * v <= pl->num_sms) S = v;
    }
    long Tw = T;
    if (S > 1 && c->opt.split_pairs && !c->fast && (op.bn_tile == 256 || op.bn_tile == 128)) {
      const long T2 = (long)op.ncls * ((m_tiles + 1) / 2) * ntn;
      int S2 = (int)((pl->num_sms / 2) / T2);
      if (S2 > nkb / 4) S2 = nkb / 4;
      if (S2 > op.bn_tile / 32) S2 = op.bn_tile / 32;
      if (c->opt.split_k >= 1 && c->opt.split_k <= S2) S2 = c->opt.split_k;
      if (S2 >= 2) { pl->cg = 2; S = S2; Tw = T2 * 2; }
      // 128-column tiles on the split path: the partial tile a CTA parks / reduces through L2 is 64 KB instead of
      // 128 KB (the split-K section is L2-bandwidth bound), at the price of a shared-memory-bound N=128 MMA phase.
      if (c->opt.split_bn128 && op.bn_tile == 256 && S2 >= 2) {
        const int ntn2 = op.cout_pad / 128;
        const long T3 = (long)op.ncls * ((m_tiles + 1) / 2) * ntn2;
        int S3 = (int)((pl->num_sms / 2) / T3);
        if (S3 > nkb / 4) S3 = nkb / 4;
        if (S3 > 4) S3 = 4;                                // 128 columns = 4 pieces of 32
        if (c->opt.split_k >= 1 && c->opt.split_k <= S3) S3 = c->opt.split_k;
        if (S3 >= 2) { op.bn_tile = 128; S = S3; Tw = T3 * 2; }
      }
    }
    pl->split_k = S;
    pl->ws_tiles = (int)Tw;                                // reduction slots: (pair-)tiles x CTAs per tile
    pl->ws_floats = S > 1 ? (size_t)Tw * S * kBM * op.bn_tile : 0;
    if (pl->ws_floats > c->splitk_ws_floats) c->splitk_ws_floats = pl->ws_floats;
    if (S > 1 && pl->ws_tiles > c->splitk_max_tiles) c->splitk_max_tiles = pl->ws_tiles;
  }
  // views + k-block table
  std::vector<ViewKey> views;
  std::vector<int4> kblk((size_t)op.ncls * nkb);
  if (pl->halo) {
    // k-block i = (input group i / 9, tap i % 9); entry = {-, K column of the weight tile, dy + 1, dx + 1}
    const int src = op.taps[0][0].src, groups = op.src[src].cin / kBK;
    views.push_back(ViewKey{src, 1, 0, 0});
    for (int i = 0; i < nkb; ++i) {
      const int g = i / 9, t = i % 9;
      kblk[i] = make_int4(0, (t * groups + g) * kBK, op.taps[0][t].ty + 1, op.taps[0][t].tx + 1);
    }
  }
  for (int cls = 0; cls < op.ncls && !pl->halo; ++cls) {
    int kb = 0;
    for (int t = 0; t < op.ntaps; ++t) {
      const Tap& tp = op.taps[cls][t];
      const int s = op.src[tp.src].s;
      ViewKey vk{tp.src, s, 0, 0};
      int dy = tp.ty, dx = tp.tx;
      if (s == 2) {
        vk.qy = ((tp.ty % 2) + 2) % 2; vk.qx = ((tp.tx % 2) + 2) % 2;
        dy = floordiv2(tp.ty); dx = floordiv2(tp.tx);
      }
      int vi = -1;
      for (size_t i = 0; i < views.size(); ++i)
        if (views[i] == vk) vi = (int)i;
      if (vi < 0) { views.push_back(vk); vi = (int)views.size() - 1; }
      const int cin = op.src[tp.src].cin;
      if (cin % kBK) { c->err = "cin not a multiple of 64: " + op.name; return IDC_ERR_ARG; }
      for (int c0 = 0; c0 < cin; c0 += kBK) kblk[(size_t)cls * nkb + kb++] = make_int4(vi * 2, c0, dy, dx);
    }
    if (kb != nkb) { c->err = "k-block count mismatch: " + op.name; return IDC_ERR_ARG; }
  }
  // A tensor maps
  std::vector<CUtensorMap> amaps(views.size() * 2);
  for (size_t i = 0; i < views.size(); ++i) {
    const ViewKey& vk = views[i];
    const ActBuf& b = c->bufs[op.src[vk.src].buf];
    const int Hv = (b.H - vk.qy + vk.s - 1) / vk.s, Wv = (b.W - vk.qx + vk.s - 1) / vk.s;
    for (int part = 0; part < 2; ++part) {
      char* base = (char*)(part == 0 ? b.p0 : b.p1);
      if (!base) { amaps[i * 2 + part] = amaps[i * 2]; continue; }  // fast mode: lo unused
      base += ((size_t)vk.qy * b.W + vk.qx) * b.C * sizeof(__half);
      cuuint64_t dims[4] = {(cuuint64_t)b.C, (cuuint64_t)Wv, (cuuint64_t)Hv, (cuuint64_t)c->max_n};
      cuuint64_t strides[3] = {(cuuint64_t)vk.s * b.C * 2, (cuuint64_t)vk.s * b.W * b.C * 2,
                               (cuuint64_t)b.H * b.W * b.C * 2};
      cuuint32_t box[4] = {(cuuint32_t)kBK, (cuuint32_t)(pl->halo ? kHaloW : op.wbox),
                           (cuuint32_t)(pl->halo ? kHaloH : op.hbox * pl->mt), 1};
      cuuint32_t estr[4] = {1, 1, 1, 1};
      CUresult r = enc(&amaps[i * 2 + part], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) {
        char msg[256];
        snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled(A) failed (%d) for op %s view %zu", (int)r, op.name.c_str(), i);
        c->err = msg;
        return IDC_ERR_CUDA;
      }
    }
  }
  // B tensor maps: [ncls*cout_pad rows][K] FP16, K-major
  for (int part = 0; part < 2; ++part) {
    cuuint64_t dims[2] = {(cuuint64_t)op.K, (cuuint64_t)op.ncls * op.cout_pad};
    cuuint64_t strides[1] = {(cuuint64_t)op.K * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)(op.bn_tile / pl->cg)};   // pairs: each CTA loads half of the weight tile
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(part == 0 ? &pl->bmap_hi : &pl->bmap_lo, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                     part == 0 ? (void*)op.w_hi : (void*)op.w_lo, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      char msg[256];
      snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled(B) failed (%d) for op %s", (int)r, op.name.c_str());
      c->err = msg;
      return IDC_ERR_CUDA;
    }
  }
  if (cudaMalloc(&pl->d_amaps, amaps.size() * sizeof(CUtensorMap)) != cudaSuccess ||
      cudaMalloc(&pl->d_kblk, kblk.size() * sizeof(int4)) != cudaSuccess) {
    c->err = "cudaMalloc failed in umma_plan_op";
    return IDC_ERR_CUDA;
  }
  cudaMemcpy(pl->d_amaps, amaps.data(), amaps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice);
  cudaMemcpy(pl->d_kblk, kblk.data(), kblk.size() * sizeof(int4), cudaMemcpyHostToDevice);

  UmmaParams& q = pl->prm;
  q.amaps = pl->d_amaps; q.n_amaps = (int)amaps.size(); q.kblk = pl->d_kblk; q.nkb = nkb; q.ncls = op.ncls;
  q.halo_groups = pl->halo ? nkb / 9 : 0;
  {
    // chunk_kb: k-blocks summed inside the tensor core before the FP32 round-to-nearest add.
    // 1 is the most accurate (1.5e-4 ab error end to end, 3.4e-4 with 2 everywhere -- profiles/).
    // Draining a chunk costs ~8 serial TMEM round trips (~1600 cycles for 128 columns per thread), about
    // one k-block of MMA time at 256 output columns per CTA tile; the Cout<=128 layers have short K
    // (few chunks per tile to amortise the tile epilogue), so they use 2 -> 2.1e-4 end to end.
    // (the rule follows the layer's width, not the tile's: the 128-column tiles of the split-K path keep chunk 1)
    const int natural = (op.cout_pad % 256 == 0) ? 256 : (op.cout_pad % 192 == 0) ? 192 : (op.cout_pad % 128 == 0) ? 128 : 64;
    int g = c->fast ? 4 : (natural <= 128 ? 2 : 1);
    if (c->opt.chunk_kb >= 1) g = c->opt.chunk_kb;
    q.chunk_kb = g;
  }
  q.tiles_y = ceil_div(op.Hl, op.hbox * pl->mt); q.tiles_x = ceil_div(op.Wl, op.wbox);
  q.n_tiles_n = op.cout_pad / op.bn_tile;
  q.hbox = op.hbox; q.wbox = op.wbox;
  q.wshift = 0;
  while ((1 << q.wshift) < op.wbox) q.wshift++;
  q.Hl = op.Hl; q.Wl = op.Wl; q.cout_pad = op.cout_pad;
  q.bias = op.epi.bias; q.scale = op.epi.scale; q.shift = op.epi.shift;
  q.gadd = nullptr; q.gadd_ld = 512; q.gadd_mult = kActScale;
  q.act = op.epi.act;
  if (op.out_f32) {
    q.out_f32 = op.out_f32_ptr; q.out_ld = op.cout_pad;
  } else if (op.out_buf >= 0) {
    const ActBuf& ob = c->bufs[op.out_buf];
    q.out_hi = (__half*)ob.p0; q.out_lo = (__half*)ob.p1;
    q.Hout = ob.H; q.Wout = ob.W; q.Cout = ob.C; q.os = op.os;
  }
  if (op.fuse_out_head) { q.wout = c->wout; q.bout = c->bout; }
  q.err = c->d_err;
  q.img0 = 0;
  q.dbgbuf = nullptr;
  return IDC_OK;
}

void umma_free_op(ConvOp& op) {
  UmmaPlan* pl = static_cast<UmmaPlan*>(op.umma_plan);
  if (!pl) return;
  if (pl->d_amaps) cudaFree(pl->d_amaps);
  if (pl->d_kblk) cudaFree(pl->d_kblk);
  delete pl;
  op.umma_plan = nullptr;
}

bool umma_op_uses_split_k(const ConvOp& op) {
  const UmmaPlan* pl = static_cast<const UmmaPlan*>(op.umma_plan);
  return pl && pl->split_k > 1;
}

cudaError_t umma_run_op(Ctx* c, ConvOp& op, int n, float* out_ab_fused, float out_mult, cudaStream_t st, int img0,
                        int max_ctas) {
  UmmaPlan* pl = static_cast<UmmaPlan*>(op.umma_plan);
  if (!pl) return cudaErrorInvalidValue;
  UmmaParams prm = pl->prm;
  prm.max_ctas = (max_ctas > 0 && pl->split_k == 1) ? (max_ctas / pl->cg) * pl->cg : 0;   // split-K needs all items co-resident
  prm.img0 = img0;
  prm.n_img = img0 + n;
  if (img0 && pl->split_k > 1) return cudaErrorInvalidValue;   // image chunks are a large-batch feature
  const int m_tiles = n * prm.tiles_y * prm.tiles_x;
  prm.total_tiles = op.ncls * (pl->cg == 2 ? (m_tiles + 1) / 2 : m_tiles) * prm.n_tiles_n;
  prm.gadd = (op.epi.gadd && c->gadd_active) ? c->gvec : nullptr;
  prm.out_ab = out_ab_fused;
  prm.dbgbuf = c->dbgbuf;
  prm.split_k = pl->split_k;
  prm.ws = c->splitk_ws;
  prm.counters = c->splitk_counters;
  if (pl->split_k > 1 && (!prm.ws || !prm.counters)) return cudaErrorInvalidValue;
  prm.out_mult = out_mult;
  if (op.fuse_out_head && !out_ab_fused) return cudaErrorInvalidValue;
  c->launch_count++;
  const bool split = !c->fast;
  const bool pdl = pdl_take(c);
#define IDC_LAUNCH(BN_, MT_, CG_)                                              \
  return split ? launch_inst<BN_, MT_, CG_, true>(*pl, prm, st, pdl) : launch_inst<BN_, MT_, CG_, false>(*pl, prm, st, pdl)
  if (pl->halo) {
    if (!split) return cudaErrorInvalidValue;
    switch (op.bn_tile * 10 + pl->cg) {
      case 641: return launch_inst<64, 1, 1, true, true>(*pl, prm, st, pdl);
      case 642: return launch_inst<64, 1, 2, true, true>(*pl, prm, st, pdl);
      case 1281: return launch_inst<128, 1, 1, true, true>(*pl, prm, st, pdl);
      case 1282: return launch_inst<128, 1, 2, true, true>(*pl, prm, st, pdl);
      default: return cudaErrorInvalidValue;
    }
  }
  switch (op.bn_tile * 100 + pl->mt * 10 + pl->cg) {
    case 6411: IDC_LAUNCH(64, 1, 1);
    case 6421: IDC_LAUNCH(64, 2, 1);
    case 12811: IDC_LAUNCH(128, 1, 1);
    case 12821: IDC_LAUNCH(128, 2, 1);
    case 19211: IDC_LAUNCH(192, 1, 1);
    case 25611: IDC_LAUNCH(256, 1, 1);
    case 25612: IDC_LAUNCH(256, 1, 2);
    case 12812: IDC_LAUNCH(128, 1, 2);
    case 12822: IDC_LAUNCH(128, 2, 2);
    case 6422: IDC_LAUNCH(64, 2, 2);
    default: return cudaErrorInvalidValue;
  }
#undef IDC_LAUNCH
}

}  // namespace idc
