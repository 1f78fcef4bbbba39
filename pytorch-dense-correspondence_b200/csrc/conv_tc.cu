// tcgen05 implicit-GEMM convolution for sm_100a: every convolution of Resnet34_8s (3x3 dilated / strided, 1x1, and the
// 7x7 stem as a patch GEMM), forward, data-gradient and weight-gradient, on the 5th-generation tensor cores.
//
//   D[128 (or 256) pixels x BLOCK_N channels] (fp32, TMEM) += A[pixels x 64 ch] (smem) * B[BLOCK_N x 64 ch]^T (smem)
//
// * Activations are NHWC bf16 planes, cut into 4x16-pixel sub-tiles.  For filter tap (r,s) and 64-channel chunk c the A
//   rows of a sub-tile are ONE 4-D TMA box load at (c, w0+(s-1)*dil, h0+(r-1)*dil, n): TMA's out-of-bounds zero fill *is*
//   the convolution padding, so there is no im2col buffer and no halo logic.
// * Weights are [Cout][tap*Cin + ci] bf16 (K-major); a [BLOCK_N x 64] box per k-block.
// * Both operands land in shared memory in the 128-byte-swizzled K-major layout tcgen05.mma consumes directly.
// * Precision: DDN_PRECISION_BF16X3 keeps fp32-equivalent results by splitting every operand x = hi + lo
//   (both bf16) and issuing hi*hi + hi*lo + lo*hi into the same fp32 TMEM accumulator (3 MMAs per k-step);
//   DDN_PRECISION_BF16 issues hi*hi only.
// * Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (one thread),
//   warps 2-5 = epilogue (tcgen05.ld -> in-register 8x8 transpose -> whole 128-byte lines of fp32 NHWC global memory, fused
//   addend / BatchNorm statistics / folded inference BatchNorm).
//   smem ring of kStages {A_hi,A_lo,B_hi,B_lo} slots with full/empty mbarriers; tcgen05.commit frees slots.
// * Kernels in this file: conv_tc_kernel (every conv, single CTA or CTA pair), conv64_halo_kernel / wgrad64_halo_kernel (the
//   64-channel layer: resident weights, one halo tile per 8x16 pixels, taps read in place), wgrad_tc_kernel (weight gradient,
//   pixels as the K dimension), operand preparation (stem patches, zero insertion, weight packs + their device-side validation).
// * Every kernel starts with griddepcontrol.launch_dependents / .wait (programmatic dependent launch, common.cuh).
//
// Reference op replaced: nn.Conv2d via conv3x3 (PSD/vision/torchvision/models/resnet.py:20-37,45,48) and the
// stride-1 1x1 downsample convs (resnet.py:210-214), plus their autograd data gradient.
#include <cuda.h>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <unordered_map>

#include "conv.cuh"
#include "conv_tc.cuh"

namespace ddn {

constexpr int TC_BLOCK_K = 64;                // bf16 elements per k-block = one 128-byte swizzle row
constexpr int TC_THREADS = 192;
constexpr int TC_A_BYTES = 128 * TC_BLOCK_K * 2;   // 16 KB

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_prefetch_l2_4d(const CUtensorMap* map, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];" ::"l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// K-major, 128-byte swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp):
//   [0,14) start>>4 | [16,30) LBO>>4 (=1, unused for swizzled K-major) | [32,46) SBO>>4 (8 rows * 128 B = 1024)
//   [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// K-major descriptor for a k-block of BK bf16 per row: BK = 64 -> 128-byte rows, SWIZZLE_128B (layout 2, SBO 1024);
// BK = 32 -> 64-byte rows, SWIZZLE_64B (layout 4, SBO 512).  Canonical layouts: cute/atom/mma_traits_sm100.hpp, Major-K.
template <int BK>
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr) {
  static_assert(BK == 64 || BK == 32, "k-block must be one 128-byte or one 64-byte swizzle row");
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((8 * BK * 2) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(BK == 64 ? 2 : 4) << 61;
  return d;
}
// Instruction descriptor for kind::f16 (cute::UMMA::InstrDescriptor): fp32 accumulate, bf16 x bf16, both K-major.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// MN-major, 128-byte swizzle descriptor: LBO = byte distance between 64-element atoms along M/N, SBO = between 8-row K groups
__device__ __forceinline__ uint64_t make_mnmajor_sw128_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__host__ __device__ constexpr uint32_t make_idesc_bf16_mn(int M, int N) {   // both operands MN-major
  return make_idesc_bf16(M, N) | (1u << 15) | (1u << 16);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// Whole-warp variants: all 32 lanes run the (warp-uniform) issue loop and ONE elected lane issues the instruction.  With the loop
// uniform the descriptors live in uniform registers and an MMA costs ~3 issue slots instead of the ~9 (R2UR + ELECT loop) the
// compiler needs when a single lane runs the loop -- which matters when an MMA is only 32 tensor-core cycles (N = 64).
__device__ __forceinline__ void umma_bf16_elect(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint32_t bar) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------ the kernel
// One persistent, warp-specialised kernel serves every convolution forward and data gradient, as a single CTA per SM
// (PAIR = false: tcgen05.mma.cta_group::1, a 128-pixel x BLOCK_N tile) or as a CTA PAIR on the two SMs of a TPC
// (PAIR = true: cta_group::2, a 256-pixel x BLOCK_N tile; each CTA stages its own 128 pixels of A and HALF of the B
// rows, so per SM the shared-memory traffic per MMA flop is half that of the single-CTA tile -- the single-CTA 128x128
// bf16x3 tile is bound by exactly that traffic: 96 KB of operand reads + 64 KB of TMA writes per 768 MMA cycles).
//
// Pixels: the output is cut into 4x16-pixel SUB-TILES (one TMA box {64 ch, 16 w, 4 h, 1 n} each, 8 KB); a CTA's 128 MMA
// rows are two consecutive sub-tiles of the flattened (image, row, column) list, which may straddle image borders, so
// 60x80 feature maps lose nothing to tile rounding (8x16 tiles wasted 6.25 % of layers 3 and 4).
// Work items: `full_items` full-width tiles (spatial-major, co-slice minor: the CTAs working on the co-slices of one pixel
// tile share its A loads in L2), then the tiles of the last, partial wave cut along N into `tail_split` pieces of
// BLOCK_N / tail_split channels (own B tensor maps), so that the tail wave costs 1/tail_split of a tile time instead
// of a whole one.  Static round-robin over the items; the three roles walk the same sequence.
//
// Epilogue variants: training forward -- raw fp32 output + per-channel sum / sum of squares added to the BatchNorm
// accumulator (bn_stats.cuh), statistics finalized by the last CTA; inference -- eval-mode BN folded to
// relu(acc*scale + shift + residual), written as fp32 and / or the next conv's bf16 planes; data gradient -- + addend.
struct TcConvParams {
  float* out;            // [N,H,W,Cout] fp32 (may be null with the folded epilogue)
  const float* addend;   // optional, same shape
  int N, H, W, Cin, Cout;   // H, W: OUTPUT size
  int taps_w;            // 1 or 3 (k x k filter)
  int dil;
  int stride;            // 1, or 2 (forward only: the A tensor map then samples every other input pixel)
  int tiles_h, tiles_w;  // 4x16 sub-tiles per image
  int n_sub;             // N * tiles_h * tiles_w
  int n_co;              // Cout / BLOCK_N
  int full_items, tail_split, total_items;
  int imgs_per_group;    // BatchNorm group of image n = n / imgs_per_group
  BnFwdFinal fin;        // fin.a.acc == nullptr: no statistics
  TcBwdStats bst;        // bst.fin.a.acc != nullptr (data gradient): column sums of the BatchNorm backward that consumes `out`
  // optional folded epilogue (inference): y = relu?(acc * ep_scale[c] + ep_shift[c] + addend)
  const float* ep_scale; const float* ep_shift; int ep_relu;
  __nv_bfloat16* out_hi; __nv_bfloat16* out_lo;
};

constexpr int TC_SUB_H = 4, TC_SUB_W = 16;     // sub-tile = one TMA box = 64 MMA rows
constexpr int TC_SUB_BYTES = 64 * 128;         // 8 KB per plane

// After the call, a[0] on lane l holds the sum over the 32 lanes of column l (butterfly reduce-scatter, 31 shuffles).
__device__ __forceinline__ void warp_colsum32(float (&a)[32], int lane) {
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
    const bool up = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float keep = up ? a[i + half] : a[i];
      const float send = up ? a[i] : a[i + half];
      a[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
}
__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// ---- CTA-pair (cta_group::2) primitives.  Barrier protocol (cutlass sm100 2-SM GEMMs): both producers' TMA loads
// complete_tx on the LEADER's full barrier (address with the peer bit cleared), the leader arms it with expect_tx for both
// CTAs' bytes and the peer arrives on it remotely; the leader's tcgen05.commit multicasts to the empty / accumulator-full
// barriers of both CTAs; the epilogue warps of both CTAs arrive on the leader's accumulator-empty barrier.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;     // cute::Sm100MmaPeerBitMask: shared::cluster address of the even (leader) CTA

__device__ __forceinline__ uint32_t cluster_cta_rank() {
  uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta_rank) {   // arrive on the barrier at `bar` in CTA cta_rank
  asm volatile(
      "{\n\t"
      ".reg .b32 remote;\n\t"
      "mapa.shared::cluster.u32 remote, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [remote];\n\t"
      "}\n" ::"r"(bar), "r"(cta_rank) : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {     // arrives on `bar` (same offset) in both CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}

// In-register transpose inside each group of 8 lanes.  In: lane 8a+b holds v[4j .. 4j+3] = elements (row 8a+b, columns 4j ..
// 4j+3), j = 0..7 (what tcgen05.ld.32x32b.x32 delivers: one accumulator row per lane).  Out: v[4i .. 4i+3] = (row 8a+i, columns
// 4b .. 4b+3).  After it the 8 lanes of a group hold the 8 column quads of ONE row for every i, so a 128-bit load / store per
// lane moves whole 128-byte lines of NHWC memory (4 lines per warp instruction instead of 32 partial ones -- the row-per-lane
// epilogue was bound by exactly that), and a column sum is 8 local adds + 2 shuffle stages.  3 butterfly stages, 48 shuffles.
__device__ __forceinline__ void transpose_8x8_quads(uint32_t (&v)[32], int lane) {
#pragma unroll
  for (int k = 1; k < 8; k <<= 1) {
    const bool up = (lane & k) != 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j & k) continue;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const uint32_t send = up ? v[4 * j + t] : v[4 * (j | k) + t];
        const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, k);
        if (up) v[4 * j + t] = recv; else v[4 * (j | k) + t] = recv;
      }
    }
  }
}

struct TcItem { int sp, co0, width; };
__device__ __forceinline__ TcItem tc_item(const TcConvParams& p, int idx, int block_n) {
  int tile = idx, piece = 0, width = block_n;
  if (idx >= p.full_items) {
    const int j = idx - p.full_items;
    tile = p.full_items + j / p.tail_split;
    piece = j - (j / p.tail_split) * p.tail_split;
    width = block_n / p.tail_split;
  }
  TcItem it;
  it.sp = tile / p.n_co;
  it.co0 = (tile - it.sp * p.n_co) * block_n + piece * width;
  it.width = width;
  return it;
}
struct TcSub { int n, h0, w0; bool valid; };
__device__ __forceinline__ TcSub tc_sub(const TcConvParams& p, int st) {
  TcSub s;
  s.valid = st < p.n_sub;
  const int tw = st % p.tiles_w; const int t = st / p.tiles_w;
  const int th = t % p.tiles_h;
  s.n = s.valid ? t / p.tiles_h : p.N;        // image index N is out of bounds for TMA: zero fill, no memory traffic
  s.h0 = th * TC_SUB_H; s.w0 = tw * TC_SUB_W;
  return s;
}

template <int BLOCK_N, int NPROD, bool PAIR>   // NPROD = 1 (bf16) or 3 (bf16x3); PAIR: BLOCK_N channels per CTA PAIR
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
               const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
               const __grid_constant__ CUtensorMap tm_bt_hi, const __grid_constant__ CUtensorMap tm_bt_lo,   // tail-width B boxes
               const TcConvParams p) {
  constexpr int NSPLIT = NPROD == 3 ? 2 : 1;
  constexpr int B_ROWS = PAIR ? BLOCK_N / 2 : BLOCK_N;         // weight rows staged by one CTA for a full-width item
  constexpr int A_BYTES = 128 * TC_BLOCK_K * 2;                // 16 KB = two sub-tile boxes
  constexpr int B_BYTES = B_ROWS * TC_BLOCK_K * 2;
  constexpr int STAGE_BYTES = NSPLIT * (A_BYTES + B_BYTES);    // per CTA
  constexpr int STAGES = (192 * 1024) / STAGE_BYTES >= 8 ? 8 : (192 * 1024) / STAGE_BYTES;
  static_assert(STAGES >= 2, "pipeline needs at least two stages");
  static_assert(2 * BLOCK_N <= 512, "two accumulators must fit the 512 TMEM columns");
  constexpr int NCOLS = 2 * BLOCK_N;
  constexpr int UMMA_M = PAIR ? 256 : 128;
  constexpr int SUBS_PER_TILE = PAIR ? 4 : 2;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[STAGES];     // PAIR: used in the leader only
  __shared__ __align__(8) uint64_t empty_bar[STAGES];
  __shared__ __align__(8) uint64_t acc_full[2];
  __shared__ __align__(8) uint64_t acc_empty[2];         // PAIR: used in the leader only
  __shared__ uint32_t tmem_base_smem;
  __shared__ int s_last;
  __shared__ __align__(16) float s_part[2][2][4][BLOCK_N];            // [accumulator][sum | sum of squares][epilogue warp][column]

  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? cluster_cta_rank() : 0u;
  const bool leader = rank == 0;
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int n_workers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int cin_chunks = p.Cin / TC_BLOCK_K;
  const int num_kb = p.taps_w * p.taps_w * cin_chunks;
  const int half = p.taps_w >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&full_bar[s]), PAIR ? 2 : 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(smem_u32(&acc_full[b]), 1); mbar_init(smem_u32(&acc_empty[b]), PAIR ? 8 : 4); }
    fence_barrier_init();
    tma_prefetch_desc(&tm_a_hi); tma_prefetch_desc(&tm_b_hi); tma_prefetch_desc(&tm_bt_hi);
    if (NSPLIT == 2) { tma_prefetch_desc(&tm_a_lo); tma_prefetch_desc(&tm_b_lo); tma_prefetch_desc(&tm_bt_lo); }
  }
  if (warp == 1) {     // TMEM allocation (whole warp; PAIR: one warp of EACH CTA takes part in the paired allocation)
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "n"(NCOLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "n"(NCOLS));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
  }
  tc_fence_before();
  __syncthreads();                 // reconverge every warp before the .aligned cluster barrier
  if (PAIR) cluster_sync_all();    // the peer's barriers are initialised before anything can arrive on them
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  pdl_wait();                      // everything above overlapped the previous kernel's tail; its results are visible from here

  if (warp == 0) {
    // ===== TMA producer (PAIR: both CTAs; own two sub-tiles of A + own half of the B rows, signalled on the leader's barrier)
    if (lane == 0) {
      uint32_t g = 0;                                  // global k-block counter across items -> ring slot / phase
      for (int idx = worker; idx < p.total_items; idx += n_workers) {
        const TcItem it = tc_item(p, idx, BLOCK_N);
        const bool tail = it.width != BLOCK_N;
        const int b_rows = PAIR ? it.width / 2 : it.width;
        const int b_row0 = it.co0 + (PAIR ? (int)rank * b_rows : 0);
        const uint32_t stage_tx = (uint32_t)(NSPLIT * (A_BYTES + b_rows * TC_BLOCK_K * 2));
        const CUtensorMap* mb_hi = tail ? &tm_bt_hi : &tm_b_hi;
        const CUtensorMap* mb_lo = tail ? &tm_bt_lo : &tm_b_lo;
        const int st0 = it.sp * SUBS_PER_TILE + (PAIR ? 2 * (int)rank : 0);
        const TcSub s0 = tc_sub(p, st0), s1 = tc_sub(p, st0 + 1);
        for (int kb = 0; kb < num_kb; ++kb, ++g) {
          const int s = g % STAGES;
          mbar_wait(smem_u32(&empty_bar[s]), ((g / STAGES) & 1) ^ 1);
          const int tap = kb / cin_chunks, cc = kb - tap * cin_chunks;
          const int r = tap / p.taps_w, sx = tap - r * p.taps_w;
          const int dh = (r - half) * p.dil, dw = (sx - half) * p.dil;
          uint8_t* stg = smem + (size_t)s * STAGE_BYTES;
          const uint32_t bar = smem_u32(&full_bar[s]);
          if (PAIR) {
            if (leader) mbar_expect_tx(bar, 2 * stage_tx);           // both CTAs' bytes land on this barrier
            else mbar_arrive_cluster(bar, 0);
            tma_load_4d_pair(smem_u32(stg), &tm_a_hi, bar, cc * TC_BLOCK_K, s0.w0 * p.stride + dw, s0.h0 * p.stride + dh, s0.n);
            tma_load_4d_pair(smem_u32(stg + TC_SUB_BYTES), &tm_a_hi, bar, cc * TC_BLOCK_K, s1.w0 * p.stride + dw, s1.h0 * p.stride + dh, s1.n);
            tma_load_2d_pair(smem_u32(stg + NSPLIT * A_BYTES), mb_hi, bar, kb * TC_BLOCK_K, b_row0);
            if (NSPLIT == 2) {
              tma_load_4d_pair(smem_u32(stg + A_BYTES), &tm_a_lo, bar, cc * TC_BLOCK_K, s0.w0 * p.stride + dw, s0.h0 * p.stride + dh, s0.n);
              tma_load_4d_pair(smem_u32(stg + A_BYTES + TC_SUB_BYTES), &tm_a_lo, bar, cc * TC_BLOCK_K, s1.w0 * p.stride + dw, s1.h0 * p.stride + dh, s1.n);
              tma_load_2d_pair(smem_u32(stg + 2 * A_BYTES + B_BYTES), mb_lo, bar, kb * TC_BLOCK_K, b_row0);
            }
          } else {
            mbar_expect_tx(bar, stage_tx);
            tma_load_4d(smem_u32(stg), &tm_a_hi, bar, cc * TC_BLOCK_K, s0.w0 * p.stride + dw, s0.h0 * p.stride + dh, s0.n);
            tma_load_4d(smem_u32(stg + TC_SUB_BYTES), &tm_a_hi, bar, cc * TC_BLOCK_K, s1.w0 * p.stride + dw, s1.h0 * p.stride + dh, s1.n);
            tma_load_2d(smem_u32(stg + NSPLIT * A_BYTES), mb_hi, bar, kb * TC_BLOCK_K, b_row0);
            if (NSPLIT == 2) {
              tma_load_4d(smem_u32(stg + A_BYTES), &tm_a_lo, bar, cc * TC_BLOCK_K, s0.w0 * p.stride + dw, s0.h0 * p.stride + dh, s0.n);
              tma_load_4d(smem_u32(stg + A_BYTES + TC_SUB_BYTES), &tm_a_lo, bar, cc * TC_BLOCK_K, s1.w0 * p.stride + dw, s1.h0 * p.stride + dh, s1.n);
              tma_load_2d(smem_u32(stg + 2 * A_BYTES + B_BYTES), mb_lo, bar, kb * TC_BLOCK_K, b_row0);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: one thread (PAIR: of the leader CTA, driving both SMs' tensor cores) =====
    if (leader && lane == 0) {
      uint32_t g = 0;
      int k_it = 0;
      for (int idx = worker; idx < p.total_items; idx += n_workers, ++k_it) {
        const TcItem it = tc_item(p, idx, BLOCK_N);
        const uint32_t idesc = make_idesc_bf16(UMMA_M, it.width);
        const int buf = k_it & 1;
        mbar_wait(smem_u32(&acc_empty[buf]), ((k_it >> 1) & 1) ^ 1);      // the epilogue(s) have drained this accumulator
        tc_fence_after();
        const uint32_t acc = tmem_base + (uint32_t)(buf * BLOCK_N);
        for (int kb = 0; kb < num_kb; ++kb, ++g) {
          const int s = g % STAGES;
          mbar_wait(smem_u32(&full_bar[s]), (g / STAGES) & 1);
          tc_fence_after();
          const uint32_t stg = smem_u32(smem + (size_t)s * STAGE_BYTES);
          const uint64_t a_hi = make_kmajor_desc<TC_BLOCK_K>(stg);
          const uint64_t b_hi = make_kmajor_desc<TC_BLOCK_K>(stg + NSPLIT * A_BYTES);
          const uint64_t a_lo = make_kmajor_desc<TC_BLOCK_K>(stg + A_BYTES);
          const uint64_t b_lo = make_kmajor_desc<TC_BLOCK_K>(stg + 2 * A_BYTES + B_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BLOCK_K / 16; ++k) {
            const uint64_t adv = (uint64_t)((k * 32) >> 4);       // 16 bf16 = 32 bytes along K inside the swizzle row
            if (PAIR) {
              if (NPROD == 3) {
                umma_bf16_pair(acc, a_hi + adv, b_lo + adv, idesc, (kb | k) != 0);
                umma_bf16_pair(acc, a_lo + adv, b_hi + adv, idesc, 1);
                umma_bf16_pair(acc, a_hi + adv, b_hi + adv, idesc, 1);
              } else {
                umma_bf16_pair(acc, a_hi + adv, b_hi + adv, idesc, (kb | k) != 0);
              }
            } else {
              if (NPROD == 3) {
                umma_bf16(acc, a_hi + adv, b_lo + adv, idesc, (kb | k) != 0);
                umma_bf16(acc, a_lo + adv, b_hi + adv, idesc, 1);
                umma_bf16(acc, a_hi + adv, b_hi + adv, idesc, 1);
              } else {
                umma_bf16(acc, a_hi + adv, b_hi + adv, idesc, (kb | k) != 0);
              }
            }
          }
          if (PAIR) umma_commit_pair(smem_u32(&empty_bar[s]));    // frees the slot (in both CTAs) once these MMAs have read it
          else umma_commit(smem_u32(&empty_bar[s]));
        }
        if (PAIR) umma_commit_pair(smem_u32(&acc_full[buf]));
        else umma_commit(smem_u32(&acc_full[buf]));
      }
    }
  } else {
    // ===== epilogue warps (PAIR: of both CTAs): own 128 pixels x width channels from the local TMEM =====
    // tcgen05.ld hands every lane one accumulator ROW (pixel); transpose_8x8_quads turns that into "8 lanes = the 8 channel quads of
    // one pixel", so every global access below is a whole 128-byte line per 8 lanes and per-channel constants are one load per lane.
    const int q = warp & 3;                          // TMEM lane quarter this warp may read
    const int e = threadIdx.x - 64;                  // 0..127
    const int ga = lane >> 3, gb = lane & 7;         // after the transpose: lane 8a+b = channel quad b of rows 32(q&1) + 8a + i, i = 0..7
    const bool stats = p.fin.a.acc != nullptr;
    const bool bstats = p.bst.fin.a.acc != nullptr;
    double* const sum_acc = bstats ? p.bst.fin.a.acc : p.fin.a.acc;
    int k_it = 0;
    for (int idx = worker; idx < p.total_items; idx += n_workers, ++k_it) {
      const TcItem it = tc_item(p, idx, BLOCK_N);
      const int buf = k_it & 1;
      const int st0 = it.sp * SUBS_PER_TILE + (PAIR ? 2 * (int)rank : 0);
      const TcSub sb = tc_sub(p, st0 + (q >> 1));
      // rows 8a .. 8a+7 of this warp's half sub-tile: image row h, columns w8 .. w8 + 7
      const int h = sb.h0 + 2 * (q & 1) + (ga >> 1), w8 = sb.w0 + 8 * (ga & 1);
      const int n_ok = (sb.valid && h < p.H) ? min(8, p.W - w8) : 0;          // valid pixels among the 8 (<= 0: none)
      const size_t pix = ((size_t)(n_ok > 0 ? sb.n : 0) * p.H + (n_ok > 0 ? h : 0)) * p.W + (n_ok > 0 ? w8 : 0);
      const size_t cbase = pix * p.Cout + it.co0 + gb * 4;                     // + i * Cout + c * 32
      const int grp = n_ok > 0 ? sb.n / p.imgs_per_group : 0;
      mbar_wait(smem_u32(&acc_full[buf]), (k_it >> 1) & 1);
      tc_fence_after();
      const int n_chunks = it.width >> 5;
#pragma unroll 1
      for (int c = 0; c < n_chunks; ++c) {
        const size_t coff = cbase + c * 32;
        // the addend (residual-branch gradient) of this chunk first: its global-load latency overlaps the TMEM read
        float4 adv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
          adv[i] = (p.addend && i < n_ok) ? __ldg(reinterpret_cast<const float4*>(p.addend + coff + (size_t)i * p.Cout)) : make_float4(0.f, 0.f, 0.f, 0.f);
        // backward statistics: the pre-BatchNorm activation (and the sign plane of the block output) of the same elements
        float4 rw[8];
        uint2 yh[8];
        if (bstats) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            rw[i] = i < n_ok ? __ldg(reinterpret_cast<const float4*>(p.bst.raw + coff + (size_t)i * p.Cout)) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.bst.y_hi) yh[i] = i < n_ok ? __ldg(reinterpret_cast<const uint2*>(p.bst.y_hi + coff + (size_t)i * p.Cout)) : make_uint2(0u, 0u);
          }
        }
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BLOCK_N + c * 32), v);
        transpose_8x8_quads(v, lane);
        float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;      // column sums of this lane's 8 rows (4 channels)
        if (p.ep_scale) {        // folded BatchNorm (+ residual, ReLU): the conv output never exists un-normalised
          const float4 sc = __ldg(reinterpret_cast<const float4*>(p.ep_scale + it.co0 + c * 32 + gb * 4));
          const float4 sh = __ldg(reinterpret_cast<const float4*>(p.ep_shift + it.co0 + c * 32 + gb * 4));
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float4 f = make_float4(fmaf(__uint_as_float(v[4 * i]), sc.x, sh.x) + adv[i].x, fmaf(__uint_as_float(v[4 * i + 1]), sc.y, sh.y) + adv[i].y,
                                   fmaf(__uint_as_float(v[4 * i + 2]), sc.z, sh.z) + adv[i].z, fmaf(__uint_as_float(v[4 * i + 3]), sc.w, sh.w) + adv[i].w);
            if (p.ep_relu) { f.x = fmaxf(f.x, 0.f); f.y = fmaxf(f.y, 0.f); f.z = fmaxf(f.z, 0.f); f.w = fmaxf(f.w, 0.f); }
            if (i < n_ok) {
              if (p.out) *reinterpret_cast<float4*>(p.out + coff + (size_t)i * p.Cout) = f;
              if (p.out_hi) {
                const __nv_bfloat16 h0 = __float2bfloat16_rn(f.x), h1 = __float2bfloat16_rn(f.y), h2 = __float2bfloat16_rn(f.z), h3 = __float2bfloat16_rn(f.w);
                *reinterpret_cast<uint2*>(p.out_hi + coff + (size_t)i * p.Cout) = make_uint2(pack_bf16x2(h0, h1), pack_bf16x2(h2, h3));
                if (p.out_lo)
                  *reinterpret_cast<uint2*>(p.out_lo + coff + (size_t)i * p.Cout) =
                      make_uint2(pack_bf16x2(__float2bfloat16_rn(f.x - __bfloat162float(h0)), __float2bfloat16_rn(f.y - __bfloat162float(h1))),
                                 pack_bf16x2(__float2bfloat16_rn(f.z - __bfloat162float(h2)), __float2bfloat16_rn(f.w - __bfloat162float(h3))));
              }
            }
          }
        } else if (bstats) {
          // g = dOut * (y > 0), (sum g, sum g * xhat): what bn_colsum_kernel<1> computes, on the gradient this kernel just wrote
          const float4 mu = __ldg(reinterpret_cast<const float4*>(p.bst.mean + (size_t)grp * p.Cout + it.co0 + c * 32 + gb * 4));
          const float4 is = __ldg(reinterpret_cast<const float4*>(p.bst.invstd + (size_t)grp * p.Cout + it.co0 + c * 32 + gb * 4));
          float4 scl = make_float4(0.f, 0.f, 0.f, 0.f), be = scl;
          if (!p.bst.y_hi && p.bst.relu) {     // no residual in the forward: y > 0 <=> bn(x) > 0, the same fmaf as bn_apply_kernel
            const float4 gm = __ldg(reinterpret_cast<const float4*>(p.bst.gamma + it.co0 + c * 32 + gb * 4));
            be = __ldg(reinterpret_cast<const float4*>(p.bst.beta + it.co0 + c * 32 + gb * 4));
            scl = make_float4(gm.x * is.x, gm.y * is.y, gm.z * is.z, gm.w * is.w);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float4 g = make_float4(__uint_as_float(v[4 * i]) + adv[i].x, __uint_as_float(v[4 * i + 1]) + adv[i].y,
                                   __uint_as_float(v[4 * i + 2]) + adv[i].z, __uint_as_float(v[4 * i + 3]) + adv[i].w);
            if (i < n_ok) *reinterpret_cast<float4*>(p.out + coff + (size_t)i * p.Cout) = g;
            else g = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.bst.y_hi) {
              const uint2 hh = yh[i];
              if ((hh.x & 0x8000u) || !(hh.x & 0x7fffu)) g.x = 0.f;
              if ((hh.x & 0x80000000u) || !(hh.x & 0x7fff0000u)) g.y = 0.f;
              if ((hh.y & 0x8000u) || !(hh.y & 0x7fffu)) g.z = 0.f;
              if ((hh.y & 0x80000000u) || !(hh.y & 0x7fff0000u)) g.w = 0.f;
            } else if (p.bst.relu) {
              if (!(fmaf(rw[i].x - mu.x, scl.x, be.x) > 0.f)) g.x = 0.f;
              if (!(fmaf(rw[i].y - mu.y, scl.y, be.y) > 0.f)) g.y = 0.f;
              if (!(fmaf(rw[i].z - mu.z, scl.z, be.z) > 0.f)) g.z = 0.f;
              if (!(fmaf(rw[i].w - mu.w, scl.w, be.w) > 0.f)) g.w = 0.f;
            }
            s1.x += g.x; s1.y += g.y; s1.z += g.z; s1.w += g.w;
            s2.x = fmaf(g.x, (rw[i].x - mu.x) * is.x, s2.x); s2.y = fmaf(g.y, (rw[i].y - mu.y) * is.y, s2.y);
            s2.z = fmaf(g.z, (rw[i].z - mu.z) * is.z, s2.z); s2.w = fmaf(g.w, (rw[i].w - mu.w) * is.w, s2.w);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            // rows outside the image hold garbage (their shifted taps can read valid pixels): neither stored nor summed
            const float4 raw = i < n_ok ? make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]))
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < n_ok)
              *reinterpret_cast<float4*>(p.out + coff + (size_t)i * p.Cout) = make_float4(raw.x + adv[i].x, raw.y + adv[i].y, raw.z + adv[i].z, raw.w + adv[i].w);
            s1.x += raw.x; s1.y += raw.y; s1.z += raw.z; s1.w += raw.w;
            s2.x = fmaf(raw.x, raw.x, s2.x); s2.y = fmaf(raw.y, raw.y, s2.y); s2.z = fmaf(raw.z, raw.z, s2.z); s2.w = fmaf(raw.w, raw.w, s2.w);
          }
        }
        if (stats || bstats) {      // the other 24 rows of this warp sit in lanes b + 8, b + 16, b + 24
#pragma unroll
          for (int off = 8; off < 32; off <<= 1) {
            s1.x += __shfl_xor_sync(0xffffffffu, s1.x, off); s1.y += __shfl_xor_sync(0xffffffffu, s1.y, off);
            s1.z += __shfl_xor_sync(0xffffffffu, s1.z, off); s1.w += __shfl_xor_sync(0xffffffffu, s1.w, off);
            s2.x += __shfl_xor_sync(0xffffffffu, s2.x, off); s2.y += __shfl_xor_sync(0xffffffffu, s2.y, off);
            s2.z += __shfl_xor_sync(0xffffffffu, s2.z, off); s2.w += __shfl_xor_sync(0xffffffffu, s2.w, off);
          }
          if (ga == 0) {
            *reinterpret_cast<float4*>(&s_part[buf][0][q][c * 32 + gb * 4]) = s1;
            *reinterpret_cast<float4*>(&s_part[buf][1][q][c * 32 + gb * 4]) = s2;
          }
        }
      }
      // the accumulator is in registers / memory now: hand the TMEM buffer back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(smem_u32(&acc_empty[buf]), 0);     // 4 warps x 2 CTAs release the leader's MMA thread
        else mbar_arrive(smem_u32(&acc_empty[buf]));
      }
      if (stats || bstats) {
        asm volatile("bar.sync 1, 128;" ::: "memory");          // the 4 epilogue warps only
        // warps 0,1 hold sub-tile A, warps 2,3 sub-tile B; their images may belong to different BatchNorm groups
        const TcSub sa = tc_sub(p, st0), sbb = tc_sub(p, st0 + 1);
        const int ga_ = sa.valid ? sa.n / p.imgs_per_group : -1, gb_ = sbb.valid ? sbb.n / p.imgs_per_group : -1;
        for (int col = e; col < it.width; col += 128) {
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const float va = s_part[buf][k][0][col] + s_part[buf][k][1][col];
            const float vb = s_part[buf][k][2][col] + s_part[buf][k][3][col];
            if (ga_ >= 0 && ga_ == gb_) {
              red_add_f64(sum_acc + (size_t)(ga_ * 2 + k) * p.Cout + it.co0 + col, (double)va + (double)vb);
            } else {
              if (ga_ >= 0) red_add_f64(sum_acc + (size_t)(ga_ * 2 + k) * p.Cout + it.co0 + col, (double)va);
              if (gb_ >= 0) red_add_f64(sum_acc + (size_t)(gb_ * 2 + k) * p.Cout + it.co0 + col, (double)vb);
            }
          }
        }
        // s_part[buf] is rewritten two items later, after another bar.sync of the same 128 threads: no extra barrier needed
      }
    }
    if (stats) {      // the last CTA turns the accumulated sums into mean / invstd / running statistics
      const bool last = bn_last_cta(p.fin.a.ticket, gridDim.x, e == 0, &s_last, [] { asm volatile("bar.sync 1, 128;" ::: "memory"); });
      if (last)
        for (int c = e; c < p.Cout; c += 128) bn_fwd_finalize_channel(p.fin, c);
    } else if (bstats) {   // ... or into dgamma / dbeta and the per-group sums bn_bwd_apply_kernel reads
      const bool last = bn_last_cta(p.bst.fin.a.ticket, gridDim.x, e == 0, &s_last, [] { asm volatile("bar.sync 1, 128;" ::: "memory"); });
      if (last)
        for (int c = e; c < p.Cout; c += 128) bn_bwd_finalize_channel(p.bst.fin, c);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();      // neither CTA frees its half of the paired TMEM while the other still uses the pair
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(NCOLS));
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(NCOLS));
  }
}

// ------------------------------------------------------------------------------------------------ 64 -> 64 channels: halo tiles
// The 3x3 convolutions of layer1 (64 -> 64 channels on the 120x160 map) have the lowest arithmetic intensity of the network:
// with one TMA box per (tap, tile) every 128-pixel tile pulls 9 x 32 KB of activations and the whole 147 KB weight tensor
// through L2 -> shared memory, ~1 GB per convolution, and the kernel above runs at the L2-to-SM throughput cap (~110 us for
// a convolution with 30 us of tensor-core work).  This kernel loads every operand ONCE:
//   * the weights (9 taps x [64 co x 64 ci], hi and lo planes, 147 KB) stay resident in shared memory for the whole launch;
//   * a tile is 8 rows x 16 columns of output pixels; its 10 x 18 HALO (one TMA box per plane, out-of-bounds = padding) is
//     staged once and all 9 taps read it in place.  The tensor map has H and W swapped, so halo pixel (h, w) is shared-memory
//     row w * 10 + h: MMA row m = 8 * (m / 8) + m % 8 is output pixel (h0 + m % 8, w0 + m / 8), the 8 rows of a core-matrix
//     group are 8 consecutive halo rows, consecutive groups are 10 rows apart (SBO = 1280 B), and tap (r, s) is the same
//     window shifted by (s * 10 + r) rows.  tcgen05 applies the 128-byte swizzle to absolute shared-memory address bits, so
//     a descriptor may start at any 128-byte row of the staged tile (base-offset field 0; scripts/probe_umma_offset.cu
//     checks exactly this on the hardware).
// bf16x3 order: first the 72 MMAs that read the hi plane of the tile (hi*lo + hi*hi), then the 36 that read the lo plane, so a
// ring of 3 plane slots always has the next plane in flight.  L2 -> SM traffic per convolution: ~110 MB instead of ~1 GB.
struct TcHaloParams {
  float* out; const float* addend;
  int N, H, W;
  int tiles_h, tiles_w, n_tiles;
  int imgs_per_group;
  BnFwdFinal fin;
  TcBwdStats bst;
  const float* ep_scale; const float* ep_shift; int ep_relu;      // folded inference epilogue (see TcConvParams)
  __nv_bfloat16* out_hi; __nv_bfloat16* out_lo;
};
constexpr int HALO_TH = 8, HALO_TW = 16;
constexpr int HALO_BH = HALO_TH + 2, HALO_BW = HALO_TW + 2;
constexpr int HALO_BOX_BYTES = HALO_BH * HALO_BW * 128;                      // 23,040
constexpr int HALO_SLOT = ((HALO_BOX_BYTES + 1023) / 1024) * 1024;           // 23,552
constexpr int HALO_SLOTS = 3;
constexpr int HALO_B_TAP = 64 * 128;                                         // one tap: 64 co x 64 ci bf16
constexpr int HALO_B_PLANE = 9 * HALO_B_TAP;

__device__ __forceinline__ uint64_t make_kmajor_sw128_desc_sbo(uint32_t smem_addr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

template <int NPROD>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv64_halo_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                   const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo, const TcHaloParams p) {
  constexpr int NSPLIT = NPROD == 3 ? 2 : 1;
  constexpr int NCOLS = 128;                                // two 64-column accumulators
  constexpr uint32_t IDESC = make_idesc_bf16(128, 64);
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_b = smem;                                   // [plane][tap][64 x 128 B]
  uint8_t* smem_a = smem + NSPLIT * HALO_B_PLANE;           // HALO_SLOTS plane slots
  __shared__ __align__(8) uint64_t full_bar[HALO_SLOTS], empty_bar[HALO_SLOTS], acc_full[2], acc_empty[2], b_full;
  __shared__ uint32_t tmem_base_smem;
  __shared__ int s_last;
  __shared__ __align__(16) float s_part[2][2][4][64];

  pdl_trigger();
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // provably warp-uniform
  if (threadIdx.x == 0) {
    for (int s = 0; s < HALO_SLOTS; ++s) { mbar_init(smem_u32(&full_bar[s]), 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(smem_u32(&acc_full[b]), 1); mbar_init(smem_u32(&acc_empty[b]), 4); }
    mbar_init(smem_u32(&b_full), 1);
    fence_barrier_init();
    tma_prefetch_desc(&tm_a_hi); tma_prefetch_desc(&tm_b_hi);
    if (NSPLIT == 2) { tma_prefetch_desc(&tm_a_lo); tma_prefetch_desc(&tm_b_lo); }
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "n"(NCOLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  pdl_wait();

  auto tile_of = [&](int t, int& n, int& h0, int& w0) {
    const int tw = t % p.tiles_w; const int q = t / p.tiles_w;
    const int th = q % p.tiles_h; n = q / p.tiles_h;
    h0 = th * HALO_TH; w0 = tw * HALO_TW;
  };

  if (warp == 0) {
    if (lane == 0) {
      const uint32_t bb = smem_u32(&b_full);
      mbar_expect_tx(bb, NSPLIT * HALO_B_PLANE);
#pragma unroll 1
      for (int tap = 0; tap < 9; ++tap) {
        tma_load_2d(smem_u32(smem_b + tap * HALO_B_TAP), &tm_b_hi, bb, tap * 64, 0);
        if (NSPLIT == 2) tma_load_2d(smem_u32(smem_b + HALO_B_PLANE + tap * HALO_B_TAP), &tm_b_lo, bb, tap * 64, 0);
      }
      uint32_t g = 0;
      // the ring holds 1.5 tiles: far enough ahead for an L2 hit, not for a DRAM miss -- so the halos of the tiles two and three
      // rounds ahead are pulled into L2 by prefetches that occupy no shared memory
      constexpr int PF = 2;
      for (int j = 0; j < PF; ++j) {
        const int tp = blockIdx.x + j * gridDim.x;
        if (tp < p.n_tiles) {
          int n, h0, w0;
          tile_of(tp, n, h0, w0);
          tma_prefetch_l2_4d(&tm_a_hi, 0, h0 - 1, w0 - 1, n);
          if (NSPLIT == 2) tma_prefetch_l2_4d(&tm_a_lo, 0, h0 - 1, w0 - 1, n);
        }
      }
      for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
        int n, h0, w0;
        {
          const int tp = t + PF * gridDim.x;
          if (tp < p.n_tiles) {
            tile_of(tp, n, h0, w0);
            tma_prefetch_l2_4d(&tm_a_hi, 0, h0 - 1, w0 - 1, n);
            if (NSPLIT == 2) tma_prefetch_l2_4d(&tm_a_lo, 0, h0 - 1, w0 - 1, n);
          }
        }
        tile_of(t, n, h0, w0);
#pragma unroll
        for (int pl = 0; pl < NSPLIT; ++pl, ++g) {
          const int s = g % HALO_SLOTS;
          mbar_wait(smem_u32(&empty_bar[s]), ((g / HALO_SLOTS) & 1) ^ 1);
          const uint32_t bar = smem_u32(&full_bar[s]);
          mbar_expect_tx(bar, HALO_BOX_BYTES);
          tma_load_4d(smem_u32(smem_a + s * HALO_SLOT), pl == 0 ? &tm_a_hi : &tm_a_lo, bar, 0, h0 - 1, w0 - 1, n);   // map dims: {c, h, w, n}
        }
      }
    }
  } else if (warp == 1) {
    {   // the whole warp walks the issue loop (see umma_bf16_elect)
      mbar_wait(smem_u32(&b_full), 0);
      tc_fence_after();
      const uint64_t bd_hi = make_kmajor_desc<TC_BLOCK_K>(smem_u32(smem_b));
      const uint64_t bd_lo = make_kmajor_desc<TC_BLOCK_K>(smem_u32(smem_b + HALO_B_PLANE));
      uint32_t g = 0;
      int k_it = 0;
      for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++k_it) {
        const int buf = k_it & 1;
        mbar_wait(smem_u32(&acc_empty[buf]), ((k_it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t acc = tmem_base + (uint32_t)(buf * 64);
        // The issuing thread has 32 tensor-core cycles per N = 64 MMA: every descriptor below is `base + compile-time constant`
        // (taps and k-steps fully unrolled), ~4 instructions per MMA.
        {   // plane hi of the tile: hi*lo + hi*hi (bf16x3) or hi*hi
          const int s = g % HALO_SLOTS;
          mbar_wait(smem_u32(&full_bar[s]), (g / HALO_SLOTS) & 1);
          tc_fence_after();
          const uint64_t a0 = make_kmajor_sw128_desc_sbo(smem_u32(smem_a + s * HALO_SLOT), HALO_BH * 128);
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t ad = a0 + (uint64_t)((((tap % 3) * HALO_BH + tap / 3) * 128 + k * 32) >> 4);
              const uint64_t boff = (uint64_t)((tap * HALO_B_TAP + k * 32) >> 4);
              if (NPROD == 3) {
                umma_bf16_elect(acc, ad, bd_lo + boff, IDESC, (tap | k) != 0);
                umma_bf16_elect(acc, ad, bd_hi + boff, IDESC, 1);
              } else {
                umma_bf16_elect(acc, ad, bd_hi + boff, IDESC, (tap | k) != 0);
              }
            }
          }
          umma_commit_elect(smem_u32(&empty_bar[s]));
          ++g;
        }
        if (NPROD == 3) {   // plane lo: lo*hi
          const int s = g % HALO_SLOTS;
          mbar_wait(smem_u32(&full_bar[s]), (g / HALO_SLOTS) & 1);
          tc_fence_after();
          const uint64_t a0 = make_kmajor_sw128_desc_sbo(smem_u32(smem_a + s * HALO_SLOT), HALO_BH * 128);
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_elect(acc, a0 + (uint64_t)((((tap % 3) * HALO_BH + tap / 3) * 128 + k * 32) >> 4),
                        bd_hi + (uint64_t)((tap * HALO_B_TAP + k * 32) >> 4), IDESC, 1);
          }
          umma_commit_elect(smem_u32(&empty_bar[s]));
          ++g;
        }
        umma_commit_elect(smem_u32(&acc_full[buf]));
      }
    }
  } else {
    const int q = warp & 3;
    const int e = threadIdx.x - 64;
    const int ga = lane >> 3, gb = lane & 7;           // after the transpose: lane 8a+b holds rows 32q + 8a + i, channel quad b
    const bool stats = p.fin.a.acc != nullptr;
    const bool bstats = p.bst.fin.a.acc != nullptr;     // data gradient: column sums of the BatchNorm backward that consumes `out`
    double* const sum_acc = bstats ? p.bst.fin.a.acc : p.fin.a.acc;
    int k_it = 0;
    for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++k_it) {
      const int buf = k_it & 1;
      int n, h0, w0;
      tile_of(t, n, h0, w0);
      // MMA row m = 32q + 8a + i is output pixel (h0 + i, w0 + 4q + a): the tiles are whole (H % 8 == 0, W % 16 == 0)
      const size_t pix0 = ((size_t)n * p.H + h0) * p.W + (w0 + 4 * q + ga);
      const size_t row_stride = (size_t)p.W * 64;      // floats between (h, w) and (h + 1, w)
      float* o = p.out + pix0 * 64 + gb * 4;
      const float* ad = p.addend ? p.addend + pix0 * 64 + gb * 4 : nullptr;
      mbar_wait(smem_u32(&acc_full[buf]), (k_it >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        float4 adv[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
          adv[i] = ad ? __ldg(reinterpret_cast<const float4*>(ad + i * row_stride + c * 32)) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 rw[8];
        uint2 yh[8];
        if (bstats) {
          const size_t boff = pix0 * 64 + gb * 4 + c * 32;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            rw[i] = __ldg(reinterpret_cast<const float4*>(p.bst.raw + boff + i * row_stride));
            if (p.bst.y_hi) yh[i] = __ldg(reinterpret_cast<const uint2*>(p.bst.y_hi + boff + i * row_stride));
          }
        }
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 64 + c * 32), v);
        transpose_8x8_quads(v, lane);
        float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
        if (p.ep_scale) {        // inference: eval-mode BatchNorm folded in, + residual, ReLU; fp32 and / or the next conv's planes
          const float4 sc = __ldg(reinterpret_cast<const float4*>(p.ep_scale + c * 32 + gb * 4));
          const float4 sf = __ldg(reinterpret_cast<const float4*>(p.ep_shift + c * 32 + gb * 4));
          const size_t eoff = pix0 * 64 + gb * 4 + c * 32;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float4 f = make_float4(fmaf(__uint_as_float(v[4 * i]), sc.x, sf.x) + adv[i].x, fmaf(__uint_as_float(v[4 * i + 1]), sc.y, sf.y) + adv[i].y,
                                   fmaf(__uint_as_float(v[4 * i + 2]), sc.z, sf.z) + adv[i].z, fmaf(__uint_as_float(v[4 * i + 3]), sc.w, sf.w) + adv[i].w);
            if (p.ep_relu) { f.x = fmaxf(f.x, 0.f); f.y = fmaxf(f.y, 0.f); f.z = fmaxf(f.z, 0.f); f.w = fmaxf(f.w, 0.f); }
            if (p.out) *reinterpret_cast<float4*>(p.out + eoff + i * row_stride) = f;
            if (p.out_hi) {
              const __nv_bfloat16 h0 = __float2bfloat16_rn(f.x), h1 = __float2bfloat16_rn(f.y), h2 = __float2bfloat16_rn(f.z), h3 = __float2bfloat16_rn(f.w);
              *reinterpret_cast<uint2*>(p.out_hi + eoff + i * row_stride) = make_uint2(pack_bf16x2(h0, h1), pack_bf16x2(h2, h3));
              if (p.out_lo)
                *reinterpret_cast<uint2*>(p.out_lo + eoff + i * row_stride) =
                    make_uint2(pack_bf16x2(__float2bfloat16_rn(f.x - __bfloat162float(h0)), __float2bfloat16_rn(f.y - __bfloat162float(h1))),
                               pack_bf16x2(__float2bfloat16_rn(f.z - __bfloat162float(h2)), __float2bfloat16_rn(f.w - __bfloat162float(h3))));
            }
          }
        } else if (bstats) {      // same arithmetic as the epilogue of conv_tc_kernel / bn_colsum_kernel<1>
          const int grp = n / p.imgs_per_group;
          const float4 mu = __ldg(reinterpret_cast<const float4*>(p.bst.mean + (size_t)grp * 64 + c * 32 + gb * 4));
          const float4 is = __ldg(reinterpret_cast<const float4*>(p.bst.invstd + (size_t)grp * 64 + c * 32 + gb * 4));
          float4 scl = make_float4(0.f, 0.f, 0.f, 0.f), be = scl;
          if (!p.bst.y_hi && p.bst.relu) {
            const float4 gm = __ldg(reinterpret_cast<const float4*>(p.bst.gamma + c * 32 + gb * 4));
            be = __ldg(reinterpret_cast<const float4*>(p.bst.beta + c * 32 + gb * 4));
            scl = make_float4(gm.x * is.x, gm.y * is.y, gm.z * is.z, gm.w * is.w);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float4 g = make_float4(__uint_as_float(v[4 * i]) + adv[i].x, __uint_as_float(v[4 * i + 1]) + adv[i].y,
                                   __uint_as_float(v[4 * i + 2]) + adv[i].z, __uint_as_float(v[4 * i + 3]) + adv[i].w);
            *reinterpret_cast<float4*>(o + i * row_stride + c * 32) = g;
            if (p.bst.y_hi) {
              const uint2 hh = yh[i];
              if ((hh.x & 0x8000u) || !(hh.x & 0x7fffu)) g.x = 0.f;
              if ((hh.x & 0x80000000u) || !(hh.x & 0x7fff0000u)) g.y = 0.f;
              if ((hh.y & 0x8000u) || !(hh.y & 0x7fffu)) g.z = 0.f;
              if ((hh.y & 0x80000000u) || !(hh.y & 0x7fff0000u)) g.w = 0.f;
            } else if (p.bst.relu) {
              if (!(fmaf(rw[i].x - mu.x, scl.x, be.x) > 0.f)) g.x = 0.f;
              if (!(fmaf(rw[i].y - mu.y, scl.y, be.y) > 0.f)) g.y = 0.f;
              if (!(fmaf(rw[i].z - mu.z, scl.z, be.z) > 0.f)) g.z = 0.f;
              if (!(fmaf(rw[i].w - mu.w, scl.w, be.w) > 0.f)) g.w = 0.f;
            }
            s1.x += g.x; s1.y += g.y; s1.z += g.z; s1.w += g.w;
            s2.x = fmaf(g.x, (rw[i].x - mu.x) * is.x, s2.x); s2.y = fmaf(g.y, (rw[i].y - mu.y) * is.y, s2.y);
            s2.z = fmaf(g.z, (rw[i].z - mu.z) * is.z, s2.z); s2.w = fmaf(g.w, (rw[i].w - mu.w) * is.w, s2.w);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 raw = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
            *reinterpret_cast<float4*>(o + i * row_stride + c * 32) = make_float4(raw.x + adv[i].x, raw.y + adv[i].y, raw.z + adv[i].z, raw.w + adv[i].w);
            s1.x += raw.x; s1.y += raw.y; s1.z += raw.z; s1.w += raw.w;
            s2.x = fmaf(raw.x, raw.x, s2.x); s2.y = fmaf(raw.y, raw.y, s2.y); s2.z = fmaf(raw.z, raw.z, s2.z); s2.w = fmaf(raw.w, raw.w, s2.w);
          }
        }
        if (stats || bstats) {      // 8 rows summed locally; the other 24 rows of this warp sit in lanes b + 8, b + 16, b + 24
#pragma unroll
          for (int off = 8; off < 32; off <<= 1) {
            s1.x += __shfl_xor_sync(0xffffffffu, s1.x, off); s1.y += __shfl_xor_sync(0xffffffffu, s1.y, off);
            s1.z += __shfl_xor_sync(0xffffffffu, s1.z, off); s1.w += __shfl_xor_sync(0xffffffffu, s1.w, off);
            s2.x += __shfl_xor_sync(0xffffffffu, s2.x, off); s2.y += __shfl_xor_sync(0xffffffffu, s2.y, off);
            s2.z += __shfl_xor_sync(0xffffffffu, s2.z, off); s2.w += __shfl_xor_sync(0xffffffffu, s2.w, off);
          }
          if (ga == 0) {
            *reinterpret_cast<float4*>(&s_part[buf][0][q][c * 32 + gb * 4]) = s1;
            *reinterpret_cast<float4*>(&s_part[buf][1][q][c * 32 + gb * 4]) = s2;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&acc_empty[buf]));
      if (stats || bstats) {
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const int grp = n / p.imgs_per_group;          // a tile lies inside one image
        const int col = e & 63, k = e >> 6;            // 128 threads = 64 columns x {sum, sum of squares}
        const float s4 = s_part[buf][k][0][col] + s_part[buf][k][1][col] + s_part[buf][k][2][col] + s_part[buf][k][3][col];
        red_add_f64(sum_acc + (size_t)(grp * 2 + k) * 64 + col, (double)s4);
      }
    }
    if (bstats) {
      const bool last = bn_last_cta(p.bst.fin.a.ticket, gridDim.x, e == 0, &s_last, [] { asm volatile("bar.sync 1, 128;" ::: "memory"); });
      if (last)
        for (int c = e; c < 64; c += 128) bn_bwd_finalize_channel(p.bst.fin, c);
    } else if (stats) {
      const bool last = bn_last_cta(p.fin.a.ticket, gridDim.x, e == 0, &s_last, [] { asm volatile("bar.sync 1, 128;" ::: "memory"); });
      if (last)
        for (int c = e; c < 64; c += 128) bn_fwd_finalize_channel(p.fin, c);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(NCOLS));
  }
}

// ------------------------------------------------------------------------------------------------ weight gradient
// dW[co][tap][ci] = sum_pixels dY[pixel][co] * X[pixel + offset(tap)][ci]  as a tcgen05 GEMM with the PIXELS as the K
// dimension.  Both operands are the same NHWC bf16 planes the forward reads, consumed as MN-MAJOR UMMA operands
// (channels contiguous, pixels = K rows), so no transposed copy exists anywhere:
//   A = dY patch: 64 pixels (4x16) x 128 output channels = two TMA boxes {64 c, 16 w, 4 h, 1 n}, 8 KB each
//   B = X  patch: 64 shifted pixels x BN input channels   = BN/64 boxes at (w0+(s-1)dil, h0+(r-1)dil); OOB zero fill
//                                                            is the padding, the shift only touches the W/H coordinates
// In shared memory a box is 64 rows (pixels) of 128 swizzled bytes (64 channels): the canonical MN-major SWIZZLE_128B
// layout with SBO = 1024 B (next 8 pixels) and LBO = 8192 B (next 64 channels = next box).
// One CTA owns (128 co) x (BN ci) x (T taps of one filter row) and a contiguous range of pixel patches (split-K);
// T accumulators of BN fp32 columns live in TMEM; the epilogue adds them into dwp[tap][co][ci] with vector reds.
// Two smem rings: A (shared by the T taps of a k-block) and B (one slot per tap).
struct TcWgradParams {
  float* dwp;            // [taps][Cout][Cin] fp32, zero-filled by the caller
  int N, H, W, Cin, Cout;
  int taps_w, dil, stride;
  int tiles_h, tiles_w;  // 4x16 (output-)pixel patches per image
  int kb_per_split;      // pixel patches per CTA (grid.z splits)
};

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <int BN, int T, int NPROD>
__global__ void __launch_bounds__(TC_THREADS, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap tm_dy_hi, const __grid_constant__ CUtensorMap tm_dy_lo,
                const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
                const TcWgradParams p) {
  constexpr int NSPLIT = NPROD == 3 ? 2 : 1;
  constexpr int A_STAGE = NSPLIT * TC_A_BYTES;                 // 128 co x 64 px per plane
  constexpr int B_PLANE = BN * TC_BLOCK_K * 2;
  constexpr int B_STAGE = NSPLIT * B_PLANE;
  constexpr int SA = 2;
  constexpr int SB_RAW = (200 * 1024 - SA * A_STAGE) / B_STAGE;
  constexpr int SB = SB_RAW > 6 ? 6 : SB_RAW;
  static_assert(SB >= 2, "B ring too small");
  constexpr int NCOLS = T * BN <= 32 ? 32 : T * BN <= 64 ? 64 : T * BN <= 128 ? 128 : T * BN <= 256 ? 256 : 512;
  constexpr uint32_t IDESC = make_idesc_bf16_mn(128, BN);
  constexpr int BOX_BYTES = 64 * 128;                          // one {64 c, 16 w, 4 h} box

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + SA * A_STAGE;
  __shared__ __align__(8) uint64_t full_a[SA], empty_a[SA], full_b[SB], empty_b[SB];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_base_smem;

  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ci_tiles = p.Cin / BN;
  const int ci0 = (blockIdx.x % ci_tiles) * BN;
  const int tap_row = blockIdx.x / ci_tiles;                   // filter row r (T == taps_w) or 0
  const int co0 = blockIdx.y * 128;
  const int total_kb = p.N * p.tiles_h * p.tiles_w;
  const int kb_begin = blockIdx.z * p.kb_per_split;
  const int kb_end = min(total_kb, kb_begin + p.kb_per_split);
  const int num_kb = kb_end - kb_begin;
  const int half = p.taps_w >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < SA; ++s) { mbar_init(smem_u32(&full_a[s]), 1); mbar_init(smem_u32(&empty_a[s]), 1); }
    for (int s = 0; s < SB; ++s) { mbar_init(smem_u32(&full_b[s]), 1); mbar_init(smem_u32(&empty_b[s]), 1); }
    mbar_init(smem_u32(&tmem_full_bar), 1);
    fence_barrier_init();
    tma_prefetch_desc(&tm_dy_hi); tma_prefetch_desc(&tm_x_hi);
    if (NSPLIT == 2) { tma_prefetch_desc(&tm_dy_lo); tma_prefetch_desc(&tm_x_lo); }
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "n"(NCOLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  pdl_wait();

  if (num_kb > 0) {
    if (warp == 0) {
      if (lane == 0) {
        for (int i = 0; i < num_kb; ++i) {
          int kb = kb_begin + i;
          const int tw = kb % p.tiles_w; kb /= p.tiles_w;
          const int th = kb % p.tiles_h; const int n = kb / p.tiles_h;
          const int h0 = th * 4, w0 = tw * 16;
          const int sa = i % SA;
          mbar_wait(smem_u32(&empty_a[sa]), ((i / SA) & 1) ^ 1);
          const uint32_t bar_a = smem_u32(&full_a[sa]);
          mbar_expect_tx(bar_a, A_STAGE);
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {      // channels co0+64..127 of a 64-channel tensor are out of bounds = zeros
            tma_load_4d(smem_u32(smem_a + sa * A_STAGE + hf * BOX_BYTES), &tm_dy_hi, bar_a, co0 + 64 * hf, w0, h0, n);
            if (NSPLIT == 2)
              tma_load_4d(smem_u32(smem_a + sa * A_STAGE + TC_A_BYTES + hf * BOX_BYTES), &tm_dy_lo, bar_a, co0 + 64 * hf, w0, h0, n);
          }
#pragma unroll
          for (int t = 0; t < T; ++t) {
            const int j = i * T + t;
            const int sb = j % SB;
            mbar_wait(smem_u32(&empty_b[sb]), ((j / SB) & 1) ^ 1);
            const int r = (T == 1) ? half : tap_row;            // 1x1: the only tap; 3x3: this CTA's filter row
            const int sx = (T == 1) ? half : t;
            const int hh = h0 * p.stride + (r - half) * p.dil, ww = w0 * p.stride + (sx - half) * p.dil;
            const uint32_t bar_b = smem_u32(&full_b[sb]);
            mbar_expect_tx(bar_b, B_STAGE);
#pragma unroll
            for (int part = 0; part < BN / 64; ++part) {
              tma_load_4d(smem_u32(smem_b + sb * B_STAGE + part * BOX_BYTES), &tm_x_hi, bar_b, ci0 + 64 * part, ww, hh, n);
              if (NSPLIT == 2)
                tma_load_4d(smem_u32(smem_b + sb * B_STAGE + B_PLANE + part * BOX_BYTES), &tm_x_lo, bar_b, ci0 + 64 * part, ww, hh, n);
            }
          }
        }
      }
    } else if (warp == 1) {
      if (lane == 0) {
        for (int i = 0; i < num_kb; ++i) {
          const int sa = i % SA;
          mbar_wait(smem_u32(&full_a[sa]), (i / SA) & 1);
          const uint32_t a_addr = smem_u32(smem_a + sa * A_STAGE);
          const uint64_t a_hi = make_mnmajor_sw128_desc(a_addr, BOX_BYTES, 1024);
          const uint64_t a_lo = make_mnmajor_sw128_desc(a_addr + TC_A_BYTES, BOX_BYTES, 1024);
#pragma unroll
          for (int t = 0; t < T; ++t) {
            const int j = i * T + t;
            const int sb = j % SB;
            mbar_wait(smem_u32(&full_b[sb]), (j / SB) & 1);
            tc_fence_after();
            const uint32_t b_addr = smem_u32(smem_b + sb * B_STAGE);
            const uint64_t b_hi = make_mnmajor_sw128_desc(b_addr, BOX_BYTES, 1024);
            const uint64_t b_lo = make_mnmajor_sw128_desc(b_addr + B_PLANE, BOX_BYTES, 1024);
            const uint32_t acc = tmem_base + (uint32_t)(t * BN);
#pragma unroll
            for (int k = 0; k < TC_BLOCK_K / 16; ++k) {
              const uint64_t adv = (uint64_t)((k * 16 * 128) >> 4);     // 16 pixels = 16 rows of 128 bytes along K
              if (NPROD == 3) {
                umma_bf16(acc, a_hi + adv, b_lo + adv, IDESC, (i | k) != 0);
                umma_bf16(acc, a_lo + adv, b_hi + adv, IDESC, 1);
                umma_bf16(acc, a_hi + adv, b_hi + adv, IDESC, 1);
              } else {
                umma_bf16(acc, a_hi + adv, b_hi + adv, IDESC, (i | k) != 0);
              }
            }
            umma_commit(smem_u32(&empty_b[sb]));
          }
          umma_commit(smem_u32(&empty_a[sa]));
        }
        umma_commit(smem_u32(&tmem_full_bar));
      }
    } else {
      const int q = warp & 3;
      const int co = co0 + q * 32 + lane;
      const bool co_ok = co < p.Cout;
      mbar_wait(smem_u32(&tmem_full_bar), 0);
      tc_fence_after();
#pragma unroll 1
      for (int t = 0; t < T; ++t) {
        const int tap = (T == 1) ? 0 : tap_row * p.taps_w + t;
        float* dst = p.dwp + ((size_t)tap * p.Cout + (co_ok ? co : 0)) * p.Cin + ci0;
#pragma unroll 1
        for (int c = 0; c < BN / 32; ++c) {
          uint32_t v[32];
          tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(t * BN + c * 32), v);
          if (co_ok)
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            red_add_v4(dst + c * 32 + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        }
      }
      tc_fence_before();
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(NCOLS));
  }
}

// ------------------------------------------------------------------------------------------------ 64 -> 64 weight gradient: halo tiles
// The kernel above gives a 64 x 64 convolution (layer1) half-empty MMAs (128 accumulator rows for 64 output channels) and, with one
// X box per (tap, 64 pixels), ~1.1 GB of L2 -> shared-memory traffic per weight gradient: it runs at the L2 throughput cap, 150 us
// for 35 us of tensor-core work.  Here a CTA walks 8 x 16-pixel tiles (the geometry and the H/W-swapped tensor maps of
// conv64_halo_kernel); per tile it stages the 10 x 18 halo of X and the 8 x 16 tile of dY ONCE, and
//   * the roles are swapped: the M side is X, shifted, with TWO TAPS STACKED along M -- the second 64-channel atom of the
//     MN-major A descriptor is the same staged halo shifted by the distance between the two taps (LBO = that many 128-byte rows;
//     scripts/probe_umma_offset.cu, "MN-stack") -- and the N side is dY (64 output channels);
//   * 9 taps = 5 accumulators of [2 taps x 64 ci] x [64 co] fp32 in TMEM (the 5th pairs tap 8 with itself), kept for the whole
//     launch; K = pixels, 16 per MMA = two columns of 8 rows (SBO = 10 halo rows for X, 8 rows for dY).
// At the end each CTA adds its partial dW into dwp[tap][co][ci] (warp-coalesced fp32 reds).
struct TcWgradHaloParams {
  float* dwp;            // [9][64][64] fp32, zero-filled by the caller
  int N, H, W;
  int tiles_h, tiles_w, n_tiles;
};
constexpr int WGH_X_SLOT = HALO_SLOT;                    // 10 x 18 halo of X, one plane
constexpr int WGH_DY_BYTES = 128 * 128;                  // 8 x 16 pixels x 64 channels, one plane
constexpr int WGH_PAIRS = 5;
__host__ __device__ constexpr int wgh_tap_a(int pr) { return pr == 0 ? 0 : pr == 1 ? 6 : pr == 2 ? 4 : pr == 3 ? 2 : 8; }   // lower halo offset
__host__ __device__ constexpr int wgh_tap_b(int pr) { return pr == 0 ? 3 : pr == 1 ? 1 : pr == 2 ? 7 : pr == 3 ? 5 : 8; }
__host__ __device__ constexpr int wgh_off(int tap) { return (tap % 3) * HALO_BH + tap / 3; }       // halo row of tap (r, s) = s * 10 + r

template <int NPROD>
__global__ void __launch_bounds__(TC_THREADS, 1)
wgrad64_halo_kernel(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
                    const __grid_constant__ CUtensorMap tm_dy_hi, const __grid_constant__ CUtensorMap tm_dy_lo, const TcWgradHaloParams p) {
  constexpr int NSPLIT = NPROD == 3 ? 2 : 1;
  constexpr int STAGE = NSPLIT * (WGH_X_SLOT + WGH_DY_BYTES);
  constexpr int STAGES = 2;
  constexpr int NCOLS = 512;                                // 5 x 64 accumulator columns
  constexpr uint32_t IDESC = make_idesc_bf16_mn(128, 64);
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], done_bar;
  __shared__ uint32_t tmem_base_smem;

  pdl_trigger();
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&full_bar[s]), 1); mbar_init(smem_u32(&empty_bar[s]), 1); }
    mbar_init(smem_u32(&done_bar), 1);
    fence_barrier_init();
    tma_prefetch_desc(&tm_x_hi); tma_prefetch_desc(&tm_dy_hi);
    if (NSPLIT == 2) { tma_prefetch_desc(&tm_x_lo); tma_prefetch_desc(&tm_dy_lo); }
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "n"(NCOLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  pdl_wait();
  const int my_tiles = p.n_tiles > (int)blockIdx.x ? (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  if (warp == 0) {
    if (lane == 0) {
      int i = 0;
      for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++i) {
        const int tw = t % p.tiles_w; const int q = t / p.tiles_w;
        const int th = q % p.tiles_h, n = q / p.tiles_h;
        const int h0 = th * HALO_TH, w0 = tw * HALO_TW;
        const int s = i % STAGES;
        mbar_wait(smem_u32(&empty_bar[s]), ((i / STAGES) & 1) ^ 1);
        const uint32_t bar = smem_u32(&full_bar[s]);
        mbar_expect_tx(bar, NSPLIT * (HALO_BOX_BYTES + WGH_DY_BYTES));
        uint8_t* stg = smem + (size_t)s * STAGE;
        tma_load_4d(smem_u32(stg), &tm_x_hi, bar, 0, h0 - 1, w0 - 1, n);                               // map dims {c, h, w, n}
        tma_load_4d(smem_u32(stg + NSPLIT * WGH_X_SLOT), &tm_dy_hi, bar, 0, h0, w0, n);
        if (NSPLIT == 2) {
          tma_load_4d(smem_u32(stg + WGH_X_SLOT), &tm_x_lo, bar, 0, h0 - 1, w0 - 1, n);
          tma_load_4d(smem_u32(stg + NSPLIT * WGH_X_SLOT + WGH_DY_BYTES), &tm_dy_lo, bar, 0, h0, w0, n);
        }
      }
    }
  } else if (warp == 1) {
    // the whole warp walks the issue loop; one elected lane issues (umma_bf16_elect).  Descriptors = base + compile-time constants.
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i % STAGES;
      mbar_wait(smem_u32(&full_bar[s]), (i / STAGES) & 1);
      tc_fence_after();
      const uint32_t stg = smem_u32(smem + (size_t)s * STAGE);
      const uint32_t x_hi = stg, x_lo = stg + WGH_X_SLOT;
      const uint32_t d_hi = stg + NSPLIT * WGH_X_SLOT, d_lo = d_hi + WGH_DY_BYTES;
#pragma unroll
      for (int pr = 0; pr < WGH_PAIRS; ++pr) {
        constexpr int dummy = 0; (void)dummy;
        const int oa = wgh_off(wgh_tap_a(pr)), ob = wgh_off(wgh_tap_b(pr));
        const uint64_t a_hi0 = make_mnmajor_sw128_desc(x_hi + oa * 128, (uint32_t)(ob - oa) * 128u, HALO_BH * 128);
        const uint64_t a_lo0 = make_mnmajor_sw128_desc(x_lo + oa * 128, (uint32_t)(ob - oa) * 128u, HALO_BH * 128);
        const uint64_t b_hi0 = make_mnmajor_sw128_desc(d_hi, 1024, 1024);
        const uint64_t b_lo0 = make_mnmajor_sw128_desc(d_lo, 1024, 1024);
        const uint32_t acc = tmem_base + (uint32_t)(pr * 64);
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {                    // 16 pixels: columns 2kk, 2kk + 1 of the tile
          const uint64_t a_adv = (uint64_t)((2 * kk * HALO_BH * 128) >> 4);
          const uint64_t b_adv = (uint64_t)((kk * 16 * 128) >> 4);
          if (NPROD == 3) {
            umma_bf16_elect(acc, a_hi0 + a_adv, b_lo0 + b_adv, IDESC, (i | kk) != 0);
            umma_bf16_elect(acc, a_lo0 + a_adv, b_hi0 + b_adv, IDESC, 1);
            umma_bf16_elect(acc, a_hi0 + a_adv, b_hi0 + b_adv, IDESC, 1);
          } else {
            umma_bf16_elect(acc, a_hi0 + a_adv, b_hi0 + b_adv, IDESC, (i | kk) != 0);
          }
        }
      }
      umma_commit_elect(smem_u32(&empty_bar[s]));
    }
    umma_commit_elect(smem_u32(&done_bar));
  } else if (my_tiles > 0) {
    const int q = warp & 3;
    const int m = q * 32 + lane;                      // accumulator row = (tap of the pair: m / 64, input channel m % 64)
    const int ci = m & 63;
    mbar_wait(smem_u32(&done_bar), 0);
    tc_fence_after();
#pragma unroll 1
    for (int pr = 0; pr < WGH_PAIRS; ++pr) {
      const int tap = (m < 64) ? wgh_tap_a(pr) : wgh_tap_b(pr);
      const bool live = pr < WGH_PAIRS - 1 || m < 64;      // the last pair holds tap 8 twice
      float* dst = p.dwp + (size_t)tap * 64 * 64 + ci;     // [tap][co][ci]: + co * 64
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(pr * 64 + c * 32), v);
        if (live) {
#pragma unroll
          for (int j = 0; j < 32; ++j) atomicAdd(dst + (size_t)(c * 32 + j) * 64, __uint_as_float(v[j]));    // result unused: RED
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(NCOLS));
  }
}

// dwp[tap][co][ci] -> dw[co][ci][r][s]
__global__ void unpack_wgrad_tc_kernel(const float* __restrict__ dwp, float* __restrict__ dw, int Cout, int Cin, int taps) {
  pdl_prologue();
  const int64_t total = (int64_t)Cout * Cin * taps;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int tap = (int)(i % taps); int64_t q = i / taps;
    int ci = (int)(q % Cin); int co = (int)(q / Cin);
    dw[i] = dwp[((int64_t)tap * Cout + co) * Cin + ci];
  }
}

// The same for many convolutions in ONE launch (blockIdx.y = table entry): the network backward leaves every conv's
// [taps][Cout][Cin] accumulator in one scratch array and converts a whole gradient bucket (a residual layer) at once.
// kind 1 = stem: dW'[co][192] (k = (r*7+s)*3 + c) -> conv1.weight gradient [64][3][7][7].
__global__ void unpack_wgrad_batched_kernel(const float* __restrict__ dwp_base, float* __restrict__ grads_base, TcUnpackTable t) {
  pdl_prologue();
  const TcUnpackEntry en = t.e[blockIdx.y];
  const float* __restrict__ dwp = dwp_base + en.src_off;
  float* __restrict__ dw = grads_base + en.dst_off;
  if (en.kind == 1) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 64 * 147; i += gridDim.x * blockDim.x) {
      const int rs = i % 49, c = (i / 49) % 3, co = i / 147;
      dw[i] = dwp[co * 192 + rs * 3 + c];
    }
    return;
  }
  const int64_t total = (int64_t)en.Cout * en.Cin * en.taps;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int tap = (int)(i % en.taps); int64_t q = i / en.taps;
    int ci = (int)(q % en.Cin); int co = (int)(q / en.Cin);
    dw[i] = dwp[((int64_t)tap * en.Cout + co) * en.Cin + ci];
  }
}

// ------------------------------------------------------------------------------------------------ operand preparation
// x fp32 -> hi = bf16(x), lo = bf16(x - hi)      (n multiple of 4)
__global__ void split_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                  int64_t n4, int want_lo) {
  pdl_prologue();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
    __nv_bfloat16 h0 = __float2bfloat16_rn(v.x), h1 = __float2bfloat16_rn(v.y), h2 = __float2bfloat16_rn(v.z), h3 = __float2bfloat16_rn(v.w);
    __nv_bfloat162 a = __halves2bfloat162(h0, h1), b = __halves2bfloat162(h2, h3);
    uint2 ho; ho.x = *reinterpret_cast<uint32_t*>(&a); ho.y = *reinterpret_cast<uint32_t*>(&b);
    reinterpret_cast<uint2*>(hi)[i] = ho;
    if (want_lo) {
      __nv_bfloat162 c = __halves2bfloat162(__float2bfloat16_rn(v.x - __bfloat162float(h0)), __float2bfloat16_rn(v.y - __bfloat162float(h1)));
      __nv_bfloat162 d = __halves2bfloat162(__float2bfloat16_rn(v.z - __bfloat162float(h2)), __float2bfloat16_rn(v.w - __bfloat162float(h3)));
      uint2 lo2; lo2.x = *reinterpret_cast<uint32_t*>(&c); lo2.y = *reinterpret_cast<uint32_t*>(&d);
      reinterpret_cast<uint2*>(lo)[i] = lo2;
    }
  }
}

// w [Cout][Cin][k][k] fp32 ->  fwd:   B[co][(r*k+s)*Cin + ci]
//                             dgrad: B[ci][(r'*k+s')*Cout + co]  with (r,s) = (k-1-r', k-1-s')
__global__ void pack_weights_tc_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                       int Cout, int Cin, int k, int dgrad, int want_lo) {
  pdl_prologue();
  const int64_t total = (int64_t)Cout * Cin * k * k;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int co, ci, r, s;
    if (!dgrad) {
      ci = (int)(i % Cin); int64_t q = i / Cin;
      s = (int)(q % k); q /= k;
      r = (int)(q % k); co = (int)(q / k);
    } else {
      co = (int)(i % Cout); int64_t q = i / Cout;
      s = k - 1 - (int)(q % k); q /= k;
      r = k - 1 - (int)(q % k); ci = (int)(q / k);
    }
    float v = w[(((int64_t)co * Cin + ci) * k + r) * k + s];
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    if (want_lo) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}


// dY fp32 [N,Ho,Wo,C] -> zero-inserted bf16 planes [N,2Ho,2Wo,C]: value at (2ho,2wo), zeros at the other three positions.
// The data gradient of a stride-2 convolution is then an ordinary stride-1 convolution over these planes.
__global__ void upsample_zero_split_kernel(const float* __restrict__ dy, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                           int N, int Ho, int Wo, int C, int want_lo) {
  pdl_prologue();
  const int q = C >> 2;
  const int64_t total = (int64_t)N * Ho * Wo * q;
  const uint2 z = make_uint2(0u, 0u);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c4 = (int)(i % q); int64_t t = i / q;
    int wo = (int)(t % Wo); t /= Wo;
    int ho = (int)(t % Ho); int n = (int)(t / Ho);
    float4 v = __ldg(reinterpret_cast<const float4*>(dy) + i);
    __nv_bfloat16 h0 = __float2bfloat16_rn(v.x), h1 = __float2bfloat16_rn(v.y), h2 = __float2bfloat16_rn(v.z), h3 = __float2bfloat16_rn(v.w);
    __nv_bfloat162 a = __halves2bfloat162(h0, h1), b = __halves2bfloat162(h2, h3);
    uint2 hv; hv.x = *reinterpret_cast<uint32_t*>(&a); hv.y = *reinterpret_cast<uint32_t*>(&b);
    uint2 lv = z;
    if (want_lo) {
      __nv_bfloat162 c = __halves2bfloat162(__float2bfloat16_rn(v.x - __bfloat162float(h0)), __float2bfloat16_rn(v.y - __bfloat162float(h1)));
      __nv_bfloat162 d = __halves2bfloat162(__float2bfloat16_rn(v.z - __bfloat162float(h2)), __float2bfloat16_rn(v.w - __bfloat162float(h3)));
      lv.x = *reinterpret_cast<uint32_t*>(&c); lv.y = *reinterpret_cast<uint32_t*>(&d);
    }
    const int64_t W2 = 2 * Wo;
    const int64_t base = (((int64_t)n * 2 * Ho + 2 * ho) * W2 + 2 * wo) * q + c4;
    uint2* H = reinterpret_cast<uint2*>(hi); uint2* L = reinterpret_cast<uint2*>(lo);
    H[base] = hv; H[base + q] = z; H[base + W2 * q] = z; H[base + W2 * q + q] = z;
    if (want_lo) { L[base] = lv; L[base + q] = z; L[base + W2 * q] = z; L[base + W2 * q + q] = z; }
  }
}

// Stem: x fp32 NCHW [N,3,H,W] -> 7x7/2 patch planes [N,H1,W1,192] bf16 (k = (r*7+s)*3 + c for k < 147, zero above), so
// that conv1 becomes a GEMM with K = 192 on the tensor cores.  One block = one output row x 64 output columns: the 7 input
// rows x 133 input columns x 3 channels it needs are staged in shared memory with coalesced loads, then written out as
// 384-byte (hi) + 384-byte (lo) rows per output pixel.
constexpr int STEM_TW = 64;
constexpr int STEM_COLS = 2 * STEM_TW + 5;
__global__ void __launch_bounds__(256)
stem_patch_split_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                        int N, int H, int W, int H1, int W1, int want_lo) {
  pdl_prologue();
  __shared__ float tile[3 * 7 * (STEM_COLS + 1) + 4];
  __shared__ int koff[192];          // k -> offset of (c, r, s) inside `tile` (the + 2*px part is added per pixel); -1 = zero padding
  const int wt = blockIdx.x, ho = blockIdx.y, n = blockIdx.z;
  const int wo0 = wt * STEM_TW;
  const int h_base = 2 * ho - 3, w_base = 2 * wo0 - 3;
  for (int k = threadIdx.x; k < 192; k += blockDim.x) {
    int off = -1;
    if (k < 147) { const int c = k % 3, rs = k / 3, r = rs / 7, sx = rs - r * 7; off = (c * 7 + r) * (STEM_COLS + 1) + sx; }
    koff[k] = off;
  }
  for (int i = threadIdx.x; i < 3 * 7 * STEM_COLS; i += blockDim.x) {
    int col = i % STEM_COLS, rc = i / STEM_COLS;
    int r = rc % 7, c = rc / 7;
    int h = h_base + r, w = w_base + col;
    float v = 0.f;
    if (h >= 0 && h < H && w >= 0 && w < W) v = __ldg(x + (((int64_t)n * 3 + c) * H + h) * W + w);
    tile[(c * 7 + r) * (STEM_COLS + 1) + col] = v;
  }
  __syncthreads();
  const int npix = min(STEM_TW, W1 - wo0);
  // thread -> a fixed group of 4 consecutive k (its four tile offsets live in registers), looping over the pixels
  const int kq = threadIdx.x % 48, px0 = threadIdx.x / 48;
  const int pstep = blockDim.x / 48;            // 256 threads: 5 pixels per sweep (16 threads idle)
  if (px0 < pstep) {
    const int o0 = koff[kq * 4], o1 = koff[kq * 4 + 1], o2 = koff[kq * 4 + 2], o3 = koff[kq * 4 + 3];
    for (int px = px0; px < npix; px += pstep) {
      const int b2 = 2 * px;
      float v[4];
      v[0] = o0 >= 0 ? tile[o0 + b2] : 0.f; v[1] = o1 >= 0 ? tile[o1 + b2] : 0.f;
      v[2] = o2 >= 0 ? tile[o2 + b2] : 0.f; v[3] = o3 >= 0 ? tile[o3 + b2] : 0.f;
      const int64_t o = (((int64_t)n * H1 + ho) * W1 + wo0 + px) * 48 + kq;
      __nv_bfloat16 h0 = __float2bfloat16_rn(v[0]), h1 = __float2bfloat16_rn(v[1]), h2 = __float2bfloat16_rn(v[2]), h3 = __float2bfloat16_rn(v[3]);
      __nv_bfloat162 a = __halves2bfloat162(h0, h1), b = __halves2bfloat162(h2, h3);
      uint2 hv; hv.x = *reinterpret_cast<uint32_t*>(&a); hv.y = *reinterpret_cast<uint32_t*>(&b);
      reinterpret_cast<uint2*>(hi)[o] = hv;
      if (want_lo) {
        __nv_bfloat162 c2 = __halves2bfloat162(__float2bfloat16_rn(v[0] - __bfloat162float(h0)), __float2bfloat16_rn(v[1] - __bfloat162float(h1)));
        __nv_bfloat162 d2 = __halves2bfloat162(__float2bfloat16_rn(v[2] - __bfloat162float(h2)), __float2bfloat16_rn(v[3] - __bfloat162float(h3)));
        uint2 lv; lv.x = *reinterpret_cast<uint32_t*>(&c2); lv.y = *reinterpret_cast<uint32_t*>(&d2);
        reinterpret_cast<uint2*>(lo)[o] = lv;
      }
    }
  }
}

// conv1.weight [64][3][7][7] fp32 -> B[co][k] bf16 hi/lo with k = (r*7+s)*3 + c, zero for k in [147,192)
__global__ void stem_pack_weights_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, int want_lo) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * 192) return;
  int k = i % 192, co = i / 192;
  float v = 0.f;
  if (k < 147) { int c = k % 3, rs = k / 3; v = w[(co * 3 + c) * 49 + rs]; }
  __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  if (want_lo) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}

// dW'[co][192] -> conv1.weight gradient [64][3][7][7]
__global__ void stem_unpack_wgrad_kernel(const float* __restrict__ dwk, float* __restrict__ dw) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * 147) return;
  int rs = i % 49, c = (i / 49) % 3, co = i / 147;
  dw[i] = dwk[co * 192 + rs * 3 + c];
}

// ------------------------------------------------------------------------------------------------ weight-pack cache
// The packed bf16 weights of every conv (forward and data-gradient layouts) live in a caller-owned cache that must never be
// stale.  Staleness is decided ON THE DEVICE: every forward fingerprints the whole fp32 parameter array (two 64-bit sums
// over the raw words, one of them position-weighted: an 85 MB read, ~15 us) and the batched pack kernel re-packs only when
// the fingerprint differs from the one the packs were made from -- so a write through `.data`, a raw pointer, an optimizer
// or NCCL is caught without any host-side version bookkeeping, and an unchanged array costs three tiny launches.
__global__ void __launch_bounds__(256)
param_fingerprint_kernel(const uint32_t* __restrict__ w, int64_t n, unsigned long long* __restrict__ fp) {
  pdl_prologue();
  unsigned long long s1 = 0, s2 = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long v = __ldg(w + i);
    s1 += v;
    s2 += v * (0x9E3779B97F4A7C15ull * (unsigned long long)(i + 1) | 1ull);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
  if ((threadIdx.x & 31) == 0) { atomicAdd(fp, s1); atomicAdd(fp + 1, s2); }
}

// blockIdx.y = table entry; packs entry's conv unless the fingerprint is unchanged (fp_new == fp_old) and !force
__global__ void __launch_bounds__(256)
pack_all_kernel(const float* __restrict__ params, char* __restrict__ cache, TcPackTable t, const unsigned long long* __restrict__ fp_new,
                const unsigned long long* __restrict__ fp_old, int force, int want_lo) {
  pdl_prologue();
  if (!force && fp_new[0] == fp_old[0] && fp_new[1] == fp_old[1]) return;
  const TcPackEntry en = t.e[blockIdx.y];
  const float* __restrict__ w = params + en.w_off;
  __nv_bfloat16* __restrict__ hi = reinterpret_cast<__nv_bfloat16*>(cache + en.dst_off);
  if (en.kind == 1) {          // stem: conv1.weight [64][3][7][7] -> B[co][k], k = (r*7+s)*3 + c, zero for k in [147,192)
    __nv_bfloat16* __restrict__ lo = hi + 64 * 192;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 64 * 192; i += gridDim.x * blockDim.x) {
      const int k = i % 192, co = i / 192;
      float v = 0.f;
      if (k < 147) { const int c = k % 3, rs = k / 3; v = w[(co * 3 + c) * 49 + rs]; }
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      hi[i] = h;
      if (want_lo) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
    return;
  }
  const int Cout = en.Cout, Cin = en.Cin, k = en.k;
  const int64_t total = (int64_t)Cout * Cin * k * k;
  __nv_bfloat16* __restrict__ lo = hi + total;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int co, ci, r, s;
    if (!en.dgrad) {
      ci = (int)(i % Cin); int64_t q = i / Cin;
      s = (int)(q % k); q /= k;
      r = (int)(q % k); co = (int)(q / k);
    } else {
      co = (int)(i % Cout); int64_t q = i / Cout;
      s = k - 1 - (int)(q % k); q /= k;
      r = k - 1 - (int)(q % k); ci = (int)(q / k);
    }
    const float v = w[(((int64_t)co * Cin + ci) * k + r) * k + s];
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    if (want_lo) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

__global__ void commit_fingerprint_kernel(unsigned long long* fp_new, unsigned long long* fp_old) {
  pdl_prologue();
  if (threadIdx.x < 2) { fp_old[threadIdx.x] = fp_new[threadIdx.x]; fp_new[threadIdx.x] = 0ull; }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// Encoded tensor maps are cached: a training step encodes the same few hundred (pointer, shape, box) combinations over and
// over (the workspace plan and the weight cache keep every operand at a fixed address), ~1 us of driver time each.
struct MapKey {
  const void* base; int d0, d1, d2, d3, b0, b1, b2, sample;
  bool operator==(const MapKey& o) const {
    return base == o.base && d0 == o.d0 && d1 == o.d1 && d2 == o.d2 && d3 == o.d3 && b0 == o.b0 && b1 == o.b1 && b2 == o.b2 && sample == o.sample;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = std::hash<const void*>()(k.base);
    for (int v : {k.d0, k.d1, k.d2, k.d3, k.b0, k.b1, k.b2, k.sample}) h = h * 1000003u ^ (size_t)v;
    return h;
  }
};
static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;
static std::mutex g_maps_mu;

// `sample` = traversal stride in W and H (elementStrides): a box then spans box*sample input pixels and delivers every
// sample-th one, which is how a stride-2 convolution reads its input without a strided copy.
static int make_act_map(CUtensorMap* m, const void* base, int N, int H, int W, int C, int sample = 1) {
  const MapKey key = {base, C, W, H, N, TC_BLOCK_K, TC_SUB_W, TC_SUB_H, sample};
  {
    std::lock_guard<std::mutex> lk(g_maps_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) { *m = it->second; return 0; }
  }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_error("cuTensorMapEncodeTiled is unavailable (driver too old?)"); return DDN_EUNSUPPORTED; }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)TC_BLOCK_K, (cuuint32_t)(TC_SUB_W * sample), (cuuint32_t)(TC_SUB_H * sample), 1};
  cuuint32_t es[4] = {1, (cuuint32_t)sample, (cuuint32_t)sample, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(activations) failed: %d", (int)r); return DDN_EINVAL; }
  std::lock_guard<std::mutex> lk(g_maps_mu);
  if (g_maps.size() > 8192) g_maps.clear();
  g_maps[key] = *m;
  return 0;
}
// Halo boxes of conv64_halo_kernel: the same NHWC planes with H and W swapped in the map, {c, h, w, n}, so that a box lands in
// shared memory as [w][h][64 c] (8 consecutive rows of a pixel column form one UMMA core-matrix group).
static int make_act_map_hw(CUtensorMap* m, const void* base, int N, int H, int W, int C, int box_h, int box_w) {
  const MapKey key = {base, C, H, W, N, TC_BLOCK_K, box_h, box_w, -2};
  {
    std::lock_guard<std::mutex> lk(g_maps_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) { *m = it->second; return 0; }
  }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_error("cuTensorMapEncodeTiled is unavailable (driver too old?)"); return DDN_EUNSUPPORTED; }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)H, (cuuint64_t)W, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)W * C * 2, (cuuint64_t)C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)TC_BLOCK_K, (cuuint32_t)box_h, (cuuint32_t)box_w, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(halo activations) failed: %d", (int)r); return DDN_EINVAL; }
  std::lock_guard<std::mutex> lk(g_maps_mu);
  if (g_maps.size() > 8192) g_maps.clear();
  g_maps[key] = *m;
  return 0;
}
static int make_act_map_halo(CUtensorMap* m, const void* base, int N, int H, int W, int C) {
  return make_act_map_hw(m, base, N, H, W, C, HALO_BH, HALO_BW);
}
static int make_weight_map(CUtensorMap* m, const void* base, int rows, int K, int box_rows) {
  const MapKey key = {base, K, rows, 0, 0, TC_BLOCK_K, box_rows, 0, -1};
  {
    std::lock_guard<std::mutex> lk(g_maps_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) { *m = it->second; return 0; }
  }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_error("cuTensorMapEncodeTiled is unavailable (driver too old?)"); return DDN_EUNSUPPORTED; }
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)TC_BLOCK_K, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(weights) failed: %d", (int)r); return DDN_EINVAL; }
  std::lock_guard<std::mutex> lk(g_maps_mu);
  if (g_maps.size() > 8192) g_maps.clear();
  g_maps[key] = *m;
  return 0;
}

// layer1's 64 -> 64 3x3 convolutions, whose (output) map tiles by HALO_TH x HALO_TW, run on the halo-tile kernels
static bool tc_halo_shape(int k, int cin, int cout, int stride, int dil, int H, int W) {
  return k == 3 && cin == 64 && cout == 64 && stride == 1 && dil == 1 && H % HALO_TH == 0 && W % HALO_TW == 0;
}

template <int BN, int T, int NPROD>
static int launch_wgrad_tc(const CUtensorMap& dy_hi, const CUtensorMap& dy_lo, const CUtensorMap& x_hi, const CUtensorMap& x_lo,
                           const TcWgradParams& p, int splits, cudaStream_t st) {
  constexpr int NSPLIT = NPROD == 3 ? 2 : 1;
  constexpr int A_STAGE = NSPLIT * TC_A_BYTES, B_STAGE = NSPLIT * BN * TC_BLOCK_K * 2;
  constexpr int SB_RAW = (200 * 1024 - 2 * A_STAGE) / B_STAGE;
  constexpr int SB = SB_RAW > 6 ? 6 : SB_RAW;
  const size_t smem = (size_t)2 * A_STAGE + (size_t)SB * B_STAGE + 1024;
  static bool configured = false;
  if (!configured) {
    DDN_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel<BN, T, NPROD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int tap_rows = (T == 1) ? 1 : p.taps_w;
  dim3 grid((unsigned)((p.Cin / BN) * tap_rows), (unsigned)ceil_div(p.Cout, 128), (unsigned)splits);
  DDN_LAUNCH((wgrad_tc_kernel<BN, T, NPROD>), grid, TC_THREADS, smem, st, dy_hi, dy_lo, x_hi, x_lo, p);
  return 0;
}

// dwp[taps][Cout][Cin] += the weight gradient from the bf16 planes of x [N,H,W,Cin] and dy [N,Ho,Wo,Cout] (Ho = H/stride).
// dw != nullptr: dwp is scratch -- zero-filled here, converted to dw[Cout][Cin][k][k] (overwritten) afterwards.
// dw == nullptr: the caller zero-filled dwp and converts it later (tc_unpack_wgrads: one launch for many convs).
int tc_wgrad_planes(TcPlanes x, TcPlanes dy, float* dw, int N, int H, int W, int Cin, int Cout, int k, int stride, int dil,
                    int precision, float* dwp, cudaStream_t st) {
  const int want_lo = precision == DDN_PRECISION_BF16X3;
  const int taps = k * k;
  const int Ho = H / stride, Wo = W / stride;
  if (dw) DDN_TRY(launch_fill_zero(dwp, sizeof(float) * (size_t)taps * Cout * Cin, st));
  if (tc_halo_shape(k, Cin, Cout, stride, dil, H, W)) {
    // layer1: one halo tile of X + one tile of dY per 8x16 pixels, two taps stacked per MMA (wgrad64_halo_kernel)
    TcWgradHaloParams hp;
    hp.dwp = dwp; hp.N = N; hp.H = H; hp.W = W; hp.tiles_h = H / HALO_TH; hp.tiles_w = W / HALO_TW; hp.n_tiles = N * hp.tiles_h * hp.tiles_w;
    CUtensorMap mx_hi, mx_lo, md_hi, md_lo;
    DDN_TRY(make_act_map_halo(&mx_hi, x.hi, N, H, W, 64));
    DDN_TRY(make_act_map_halo(&mx_lo, want_lo ? x.lo : x.hi, N, H, W, 64));
    DDN_TRY(make_act_map_hw(&md_hi, dy.hi, N, H, W, 64, HALO_TH, HALO_TW));
    DDN_TRY(make_act_map_hw(&md_lo, want_lo ? dy.lo : dy.hi, N, H, W, 64, HALO_TH, HALO_TW));
    const int nsplit = want_lo ? 2 : 1;
    const size_t smem = (size_t)2 * nsplit * (WGH_X_SLOT + WGH_DY_BYTES) + 1024;
    const int grid = std::min(hp.n_tiles, num_sms());
    {
      ProfScope ps(PROF_CONV_WGRAD_TC, 2.0 * N * H * W * 64.0 * 9 * 64, st);
      if (want_lo) {
        static bool configured = false;
        if (!configured) { DDN_CUDA(cudaFuncSetAttribute(wgrad64_halo_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); configured = true; }
        DDN_LAUNCH((wgrad64_halo_kernel<3>), grid, TC_THREADS, smem, st, mx_hi, mx_lo, md_hi, md_lo, hp);
      } else {
        static bool configured = false;
        if (!configured) { DDN_CUDA(cudaFuncSetAttribute(wgrad64_halo_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); configured = true; }
        DDN_LAUNCH((wgrad64_halo_kernel<1>), grid, TC_THREADS, smem, st, mx_hi, mx_lo, md_hi, md_lo, hp);
      }
    }
    if (dw) {
      int blocks = (int)std::min<int64_t>(ceil_div((int64_t)taps * Cout * Cin, 256), 4096);
      DDN_LAUNCH(unpack_wgrad_tc_kernel, blocks, 256, 0, st, dwp, dw, Cout, Cin, taps);
    }
    return 0;
  }
  const int bn = Cin % 128 == 0 ? 128 : 64;
  CUtensorMap m_dy_hi, m_dy_lo, m_x_hi, m_x_lo;
  DDN_TRY(make_act_map(&m_dy_hi, dy.hi, N, Ho, Wo, Cout));
  DDN_TRY(make_act_map(&m_dy_lo, want_lo ? dy.lo : dy.hi, N, Ho, Wo, Cout));
  DDN_TRY(make_act_map(&m_x_hi, x.hi, N, H, W, Cin, stride));
  DDN_TRY(make_act_map(&m_x_lo, want_lo ? x.lo : x.hi, N, H, W, Cin, stride));
  TcWgradParams p;
  p.dwp = dwp; p.N = N; p.H = Ho; p.W = Wo; p.Cin = Cin; p.Cout = Cout; p.taps_w = k; p.dil = dil; p.stride = stride;
  p.tiles_h = (int)ceil_div(Ho, 4); p.tiles_w = (int)ceil_div(Wo, 16);
  const int total_kb = N * p.tiles_h * p.tiles_w;
  const int ctas_xy = (Cin / bn) * (k == 3 ? 3 : 1) * (int)ceil_div(Cout, 128);
  // split-K so that the grid is (just under) a whole number of waves: 1 CTA per SM resident, no ragged tail wave
  const int sms = num_sms();
  int waves = ctas_xy > sms ? 1 : (total_kb >= 64 * (sms / ctas_xy) ? 2 : 1);
  int splits = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)waves * sms / ctas_xy, ceil_div(total_kb, 4)));
  p.kb_per_split = (int)ceil_div(total_kb, splits);
  splits = (int)ceil_div(total_kb, p.kb_per_split);
  const double fl = 2.0 * N * Ho * Wo * (double)Cout * taps * Cin;
  {
    ProfScope ps(PROF_CONV_WGRAD_TC, fl, st);
#define WG(BNV, TV)                                                                                      \
  do {                                                                                                   \
    if (want_lo) DDN_TRY((launch_wgrad_tc<BNV, TV, 3>(m_dy_hi, m_dy_lo, m_x_hi, m_x_lo, p, splits, st))); \
    else DDN_TRY((launch_wgrad_tc<BNV, TV, 1>(m_dy_hi, m_dy_lo, m_x_hi, m_x_lo, p, splits, st)));         \
  } while (0)
    if (k == 3) { if (bn == 128) WG(128, 3); else WG(64, 3); }
    else { if (bn == 128) WG(128, 1); else WG(64, 1); }
#undef WG
  }
  if (dw) {
    int blocks = (int)std::min<int64_t>(ceil_div((int64_t)taps * Cout * Cin, 256), 4096);
    DDN_LAUNCH(unpack_wgrad_tc_kernel, blocks, 256, 0, st, dwp, dw, Cout, Cin, taps);
  }
  return 0;
}

int tc_unpack_wgrads(const TcUnpackEntry* entries, int n, const float* dwp_base, float* grads_base, cudaStream_t st) {
  for (int i0 = 0; i0 < n; i0 += TC_UNPACK_MAX) {
    TcUnpackTable t; t.n = std::min(TC_UNPACK_MAX, n - i0);
    int64_t biggest = 0;
    for (int i = 0; i < t.n; ++i) { t.e[i] = entries[i0 + i]; biggest = std::max<int64_t>(biggest, (int64_t)t.e[i].Cout * t.e[i].Cin * t.e[i].taps); }
    dim3 grid((unsigned)std::min<int64_t>(ceil_div(biggest, 256 * 4), 1024), (unsigned)t.n);
    DDN_LAUNCH(unpack_wgrad_batched_kernel, grid, 256, 0, st, dwp_base, grads_base, t);
  }
  return 0;
}

bool tc_available() { return true; }

// forward / weight-gradient coverage: 3x3 (pad == dil) or 1x1 (pad 0), stride 1 -- or stride 2 with dil 1 on even sizes
bool tc_conv_supported(int Cin, int Cout, int k, int stride, int pad, int dil, int H, int W) {
  if (Cin % 64 || Cout % 64) return false;
  if (stride == 2) { if (dil != 1 || (H & 1) || (W & 1)) return false; }
  else if (stride != 1) return false;
  if (k == 3) return pad == dil;
  if (k == 1) return pad == 0;
  return false;
}

static const size_t kMaxWeightElems = (size_t)9 * 512 * 512;
size_t tc_weight_ws_bytes() { return 2 * align_up(kMaxWeightElems * 2, 1024) + 2048; }

int tc_split(const float* x, __nv_bfloat16* hi, __nv_bfloat16* lo, int64_t n, int precision, cudaStream_t st) {
  DDN_CHECK_ARG(n % 4 == 0, "split: element count must be a multiple of 4");
  int64_t n4 = n / 4;
  int blocks = (int)std::min<int64_t>(ceil_div(n4, 256), (int64_t)num_sms() * 8);
  DDN_LAUNCH(split_bf16_kernel, blocks, 256, 0, st, x, hi, lo, n4, precision == DDN_PRECISION_BF16X3 ? 1 : 0);
  return 0;
}

int tc_pack_weights(const float* w_oihw, __nv_bfloat16* hi, __nv_bfloat16* lo, int Cout, int Cin, int k, int dgrad, int precision,
                    cudaStream_t st) {
  const size_t wel = (size_t)Cout * Cin * k * k;
  int wblocks = (int)std::min<int64_t>(ceil_div((int64_t)wel, 256), 4096);
  DDN_LAUNCH(pack_weights_tc_kernel, wblocks, 256, 0, st, w_oihw, hi, lo, Cout, Cin, k, dgrad, precision == DDN_PRECISION_BF16X3 ? 1 : 0);
  return 0;
}

int tc_upsample_zero_split(const float* dy, __nv_bfloat16* hi, __nv_bfloat16* lo, int N, int Ho, int Wo, int C, int precision,
                           cudaStream_t st) {
  int64_t total = (int64_t)N * Ho * Wo * (C / 4);
  int blocks = (int)std::min<int64_t>(ceil_div(total, 256), (int64_t)num_sms() * 8);
  DDN_LAUNCH(upsample_zero_split_kernel, blocks, 256, 0, st, dy, hi, lo, N, Ho, Wo, C, precision == DDN_PRECISION_BF16X3 ? 1 : 0);
  return 0;
}

int tc_stem_patches(const float* x_nchw, __nv_bfloat16* hi, __nv_bfloat16* lo, int N, int H, int W, int precision, cudaStream_t st) {
  const int H1 = (H - 1) / 2 + 1, W1 = (W - 1) / 2 + 1;
  DDN_CHECK_ARG(N <= 65535 && H1 <= 65535, "stem: batch / height too large for the launch grid");
  dim3 grid((unsigned)ceil_div(W1, STEM_TW), (unsigned)H1, (unsigned)N);
  DDN_LAUNCH(stem_patch_split_kernel, grid, 256, 0, st, x_nchw, hi, lo, N, H, W, H1, W1, precision == DDN_PRECISION_BF16X3 ? 1 : 0);
  return 0;
}

template <int BLOCK_N, int NPROD, bool PAIR>
static int launch_conv_tc(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo,
                          const CUtensorMap& bt_hi, const CUtensorMap& bt_lo, const TcConvParams& p, int workers, cudaStream_t st) {
  constexpr int NSPLIT = NPROD == 3 ? 2 : 1;
  constexpr int B_ROWS = PAIR ? BLOCK_N / 2 : BLOCK_N;
  constexpr int STAGE_BYTES = NSPLIT * (128 * TC_BLOCK_K * 2 + B_ROWS * TC_BLOCK_K * 2);
  constexpr int STAGES = (192 * 1024) / STAGE_BYTES >= 8 ? 8 : (192 * 1024) / STAGE_BYTES;
  const size_t smem = (size_t)STAGES * STAGE_BYTES + 1024;
  static bool configured = false;
  if (!configured) {
    DDN_CUDA(cudaFuncSetAttribute(conv_tc_kernel<BLOCK_N, NPROD, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  DDN_LAUNCH_CLUSTER((conv_tc_kernel<BLOCK_N, NPROD, PAIR>), PAIR ? 2 * workers : workers, PAIR ? 2 : 1, TC_THREADS, smem, st,
                     a_hi, a_lo, b_hi, b_lo, bt_hi, bt_lo, p);
  return 0;
}

template <int NPROD>
static int launch_conv64_halo(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo,
                              const TcHaloParams& p, cudaStream_t st) {
  constexpr int NSPLIT = NPROD == 3 ? 2 : 1;
  const size_t smem = (size_t)NSPLIT * HALO_B_PLANE + (size_t)HALO_SLOTS * HALO_SLOT + 1024;
  static bool configured = false;
  if (!configured) {
    DDN_CUDA(cudaFuncSetAttribute(conv64_halo_kernel<NPROD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int grid = std::min(p.n_tiles, num_sms());
  DDN_LAUNCH((conv64_halo_kernel<NPROD>), grid, TC_THREADS, smem, st, a_hi, a_lo, b_hi, b_lo, p);
  return 0;
}

// out[N,Ho,Wo,gout] = conv(planes of in[N,H,W,gin]) (+ addend).
//   dgrad = 0: forward (gin = Cin, gout = Cout, Ho = H/stride).
//   dgrad = 1: data gradient, stride 1 only (`in` = dY planes with Cout channels, out = dX with Cin channels; Cin/Cout are
//              those of the ORIGINAL conv).
//   wpk != nullptr: weights are already packed [gout][k*k*gin] bf16 hi/lo; else they are packed from w_oihw into `wws`.
//   stats (forward only): per-channel sum / sum of squares of the output go to stats->a, and the kernel's last CTA writes
//              the BatchNorm statistics described by *stats; groups = BatchNorm groups in the batch.
//   bst (data gradient only): the gradient written to `out` is the dY of a BatchNorm whose column sums (sum g, sum g*xhat,
//              g = dY * relu mask) are accumulated by the epilogue; the last CTA finalizes them like bn_colsum_kernel<1>.
int tc_conv_planes(TcPlanes in, const float* w_oihw, const TcPlanes* wpk, float* out, const float* addend, const BnFwdFinal* stats,
                   int N, int H, int W, int Cin, int Cout, int k, int stride, int dil, int dgrad, int precision,
                   void* wws, size_t wws_bytes, cudaStream_t st, const TcFoldedEpilogue* ep, const TcBwdStats* bst) {
  DDN_CHECK_ARG(stride == 1 || !dgrad, "the strided data gradient goes through zero-inserted planes (stride 1 here)");
  const int Ho = H / stride, Wo = W / stride;
  const double fl = 2.0 * N * Ho * Wo * (double)Cout * k * k * Cin;
  const int gin = dgrad ? Cout : Cin, gout = dgrad ? Cin : Cout;
  const int want_lo = precision == DDN_PRECISION_BF16X3;
  const __nv_bfloat16* b_hi; const __nv_bfloat16* b_lo;
  if (wpk) {
    b_hi = wpk->hi; b_lo = wpk->lo;
  } else {
    const size_t wel = (size_t)Cout * Cin * k * k;
    const size_t w_b = align_up(kMaxWeightElems * 2, 1024);
    DDN_CHECK_ARG(wws != nullptr && wel <= kMaxWeightElems, "tc weight staging missing or weight tensor too large");
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<uintptr_t>(wws), 1024));
    if ((size_t)(base - (char*)wws) + 2 * w_b > wws_bytes) { set_error("tcgen05 weight staging too small"); return DDN_EWORKSPACE; }
    __nv_bfloat16* ph = (__nv_bfloat16*)base; __nv_bfloat16* pl = (__nv_bfloat16*)(base + w_b);
    int wblocks = (int)std::min<int64_t>(ceil_div((int64_t)wel, 256), 4096);
    DDN_LAUNCH(pack_weights_tc_kernel, wblocks, 256, 0, st, w_oihw, ph, pl, Cout, Cin, k, dgrad, want_lo);
    b_hi = ph; b_lo = pl;
  }
  if (tc_halo_shape(k, gin, gout, stride, dil, Ho, Wo)) {
    // 64 -> 64 channels (layer1): resident weights + one halo tile per 8x16 output pixels (conv64_halo_kernel)
    TcHaloParams hp;
    memset(&hp, 0, sizeof(hp));
    if (ep) {
      DDN_CHECK_ARG(!dgrad && !stats && !bst && ep->scale && ep->shift && (out || ep->out_hi), "folded epilogue: forward only, needs scale/shift and an output");
      hp.ep_scale = ep->scale; hp.ep_shift = ep->shift; hp.ep_relu = ep->relu; hp.out_hi = ep->out_hi; hp.out_lo = want_lo ? ep->out_lo : nullptr;
    } else {
      DDN_CHECK_ARG(out != nullptr, "conv output pointer is null");
    }
    hp.out = out; hp.addend = addend; hp.N = N; hp.H = Ho; hp.W = Wo;
    hp.tiles_h = Ho / HALO_TH; hp.tiles_w = Wo / HALO_TW; hp.n_tiles = N * hp.tiles_h * hp.tiles_w;
    hp.imgs_per_group = N;
    if (stats) {
      DDN_CHECK_ARG(!dgrad && stats->G >= 1 && stats->G <= BN_MAX_GROUPS && N % stats->G == 0 && stats->C == 64, "bad BatchNorm statistics request");
      hp.fin = *stats;
      hp.imgs_per_group = N / stats->G;
    }
    if (bst) {
      DDN_CHECK_ARG(dgrad && !stats && bst->raw && bst->mean && bst->invstd && bst->fin.a.acc && bst->fin.G >= 1 && bst->fin.G <= BN_MAX_GROUPS &&
                    N % bst->fin.G == 0 && bst->fin.C == 64 && (bst->y_hi || !bst->relu || (bst->gamma && bst->beta)),
                    "bad BatchNorm backward-statistics request");
      hp.bst = *bst;
      hp.imgs_per_group = N / bst->fin.G;
    }
    CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
    DDN_TRY(make_act_map_halo(&ma_hi, in.hi, N, H, W, 64));
    DDN_TRY(make_act_map_halo(&ma_lo, want_lo ? in.lo : in.hi, N, H, W, 64));
    DDN_TRY(make_weight_map(&mb_hi, b_hi, 64, 9 * 64, 64));
    DDN_TRY(make_weight_map(&mb_lo, want_lo ? b_lo : b_hi, 64, 9 * 64, 64));
    ProfScope ps(dgrad ? PROF_CONV_DGRAD_TC : PROF_CONV_FWD_TC, fl, st);
    return want_lo ? launch_conv64_halo<3>(ma_hi, ma_lo, mb_hi, mb_lo, hp, st) : launch_conv64_halo<1>(ma_hi, ma_lo, mb_hi, mb_lo, hp, st);
  }
  // CTA pairs (256 x 256 tiles) for Cout % 256 == 0.  Pairing Cout = 128 as 256 x 128 tiles measured no faster than single CTAs
  // (DESIGN.md §8).
  const bool pair = gout % 256 == 0;
  const int block_n = pair ? 256 : gout % 128 == 0 ? 128 : 64;
  TcConvParams p;
  memset(&p, 0, sizeof(p));
  p.out = out; p.addend = addend; p.N = N; p.H = Ho; p.W = Wo; p.Cin = gin; p.Cout = gout; p.taps_w = k; p.dil = dil;
  p.stride = stride;
  p.tiles_h = (int)ceil_div(Ho, TC_SUB_H); p.tiles_w = (int)ceil_div(Wo, TC_SUB_W);
  p.n_sub = N * p.tiles_h * p.tiles_w;
  p.n_co = gout / block_n;
  const int subs_per_tile = pair ? 4 : 2;
  const int tiles = (int)ceil_div(p.n_sub, subs_per_tile) * p.n_co;
  const int workers_max = pair ? num_sms() / 2 : num_sms();
  // the tiles of the last, partial wave are cut along N so that the tail costs a fraction of a tile time
  const int rem = tiles % workers_max;
  const int min_width = pair ? 64 : 32;
  int split = 1;
  if (rem)
    while (split * 2 <= 8 && block_n / (split * 2) >= min_width && rem * split * 2 <= workers_max) split *= 2;
  p.full_items = tiles - rem; p.tail_split = split; p.total_items = p.full_items + rem * split;
  if (split == 1) { p.full_items = tiles; p.total_items = tiles; }
  const int workers = std::min(p.total_items, workers_max);
  p.imgs_per_group = N;
  if (stats) {
    DDN_CHECK_ARG(!dgrad && !ep && stats->G >= 1 && stats->G <= BN_MAX_GROUPS && N % stats->G == 0, "bad BatchNorm statistics request");
    p.fin = *stats;
    p.imgs_per_group = N / stats->G;
  }
  if (bst) {
    DDN_CHECK_ARG(dgrad && !ep && !stats && bst->raw && bst->mean && bst->invstd && bst->fin.a.acc && bst->fin.G >= 1 &&
                  bst->fin.G <= BN_MAX_GROUPS && N % bst->fin.G == 0 && bst->fin.C == gout && (bst->y_hi || !bst->relu || (bst->gamma && bst->beta)),
                  "bad BatchNorm backward-statistics request");
    p.bst = *bst;
    p.imgs_per_group = N / bst->fin.G;
  }
  if (ep) {
    DDN_CHECK_ARG(!dgrad && !stats && ep->scale && ep->shift && (out || ep->out_hi), "folded epilogue: forward only, needs scale/shift and an output");
    p.ep_scale = ep->scale; p.ep_shift = ep->shift; p.ep_relu = ep->relu; p.out_hi = ep->out_hi; p.out_lo = want_lo ? ep->out_lo : nullptr;
  } else {
    DDN_CHECK_ARG(out != nullptr, "conv output pointer is null");
  }
  const int b_rows = pair ? block_n / 2 : block_n;
  const int bt_rows = b_rows / split;
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo, mt_hi, mt_lo;
  DDN_TRY(make_act_map(&ma_hi, in.hi, N, H, W, gin, stride));
  DDN_TRY(make_act_map(&ma_lo, want_lo ? in.lo : in.hi, N, H, W, gin, stride));
  DDN_TRY(make_weight_map(&mb_hi, b_hi, gout, k * k * gin, b_rows));
  DDN_TRY(make_weight_map(&mb_lo, want_lo ? b_lo : b_hi, gout, k * k * gin, b_rows));
  DDN_TRY(make_weight_map(&mt_hi, b_hi, gout, k * k * gin, bt_rows));
  DDN_TRY(make_weight_map(&mt_lo, want_lo ? b_lo : b_hi, gout, k * k * gin, bt_rows));
  ProfScope ps(dgrad ? PROF_CONV_DGRAD_TC : PROF_CONV_FWD_TC, fl, st);   // times the MMA kernel only
#define CONV_TC(BN, PR)                                                                                                       \
  (want_lo ? launch_conv_tc<BN, 3, PR>(ma_hi, ma_lo, mb_hi, mb_lo, mt_hi, mt_lo, p, workers, st)                               \
           : launch_conv_tc<BN, 1, PR>(ma_hi, ma_lo, mb_hi, mb_lo, mt_hi, mt_lo, p, workers, st))
  if (pair) return CONV_TC(256, true);
  if (block_n == 128) return CONV_TC(128, false);
  return CONV_TC(64, false);
#undef CONV_TC
}

// data gradient of a stride-2 conv: zero-insert dY [N,H/2,W/2,Cout] into `up` planes [N,H,W,Cout], then a stride-1 dgrad
int tc_dgrad_strided(const float* dy_f32, TcPlanes up, const float* w_oihw, const TcPlanes* w_packed, float* dx, const float* addend,
                     int N, int H, int W, int Cin, int Cout, int k, int precision, void* wws, size_t wws_bytes, cudaStream_t st,
                     const TcBwdStats* bst) {
  DDN_TRY(tc_upsample_zero_split(dy_f32, const_cast<__nv_bfloat16*>(up.hi), const_cast<__nv_bfloat16*>(up.lo), N, H / 2, W / 2, Cout,
                                 precision, st));
  return tc_conv_planes(up, w_oihw, w_packed, dx, addend, nullptr, N, H, W, Cin, Cout, k, 1, 1, 1, precision, wws, wws_bytes, st, nullptr, bst);
}

// ---- stem (conv1 7x7/2, Cin = 3) as a K = 192 GEMM over patch planes
int tc_stem_pack_weights(const float* w_conv1, __nv_bfloat16* hi, __nv_bfloat16* lo, int precision, cudaStream_t st) {
  DDN_LAUNCH(stem_pack_weights_kernel, (64 * 192 + 255) / 256, 256, 0, st, w_conv1, hi, lo, precision == DDN_PRECISION_BF16X3 ? 1 : 0);
  return 0;
}
int tc_stem_forward(TcPlanes patches, const float* w_conv1, const TcPlanes* w_packed, float* raw, const BnFwdFinal* stats, int N, int H1,
                    int W1, int precision, void* wws, size_t wws_bytes, cudaStream_t st) {
  TcPlanes wpk;
  if (w_packed) wpk = *w_packed;
  else {
    char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<uintptr_t>(wws), 1024));
    DDN_CHECK_ARG((size_t)(base - (char*)wws) + 2 * 64 * 192 * 2 + 1024 <= wws_bytes, "weight staging too small");
    __nv_bfloat16* ph = (__nv_bfloat16*)base; __nv_bfloat16* pl = (__nv_bfloat16*)(base + align_up((size_t)64 * 192 * 2, 1024));
    DDN_TRY(tc_stem_pack_weights(w_conv1, ph, pl, precision, st));
    wpk.hi = ph; wpk.lo = pl;
  }
  return tc_conv_planes(patches, nullptr, &wpk, raw, nullptr, stats, N, H1, W1, 192, 64, 1, 1, 1, 0, precision, wws, wws_bytes, st);
}

// d conv1.weight [64,3,7,7] from the patch planes and the planes of d(raw stem output).
// dw_conv1 != nullptr: immediate (scratch: 2 x 64*192 floats); else dwp_deferred [64][192] (pre-zeroed) is left for tc_unpack_wgrads.
int tc_stem_wgrad(TcPlanes patches, TcPlanes dy, float* dw_conv1, int N, int H1, int W1, int precision, float* scratch, cudaStream_t st) {
  if (!dw_conv1) return tc_wgrad_planes(patches, dy, nullptr, N, H1, W1, 192, 64, 1, 1, 1, precision, scratch, st);
  float* dwp = scratch; float* dwk = scratch + 64 * 192;
  DDN_TRY(tc_wgrad_planes(patches, dy, dwk, N, H1, W1, 192, 64, 1, 1, 1, precision, dwp, st));
  DDN_LAUNCH(stem_unpack_wgrad_kernel, (64 * 147 + 255) / 256, 256, 0, st, dwk, dw_conv1);
  return 0;
}

// (re)packs every table entry into `cache` when the device-side fingerprint of params[0..n_params) differs from the one
// stored at `fp_old` (or `force`): three launches, no host synchronisation.  fp_new / fp_old: 2 x uint64 each, fp_new zero.
int tc_pack_all(const float* params, int64_t n_params, char* cache, const TcPackEntry* entries, int n, unsigned long long* fp_new,
                unsigned long long* fp_old, int force, int precision, cudaStream_t st) {
  DDN_CHECK_ARG(n >= 1 && n <= TC_PACK_MAX, "pack table too large");
  TcPackTable t; t.n = n;
  for (int i = 0; i < n; ++i) t.e[i] = entries[i];
  DDN_LAUNCH(param_fingerprint_kernel, num_sms() * 2, 256, 0, st, reinterpret_cast<const uint32_t*>(params), n_params, fp_new);
  dim3 grid(32, (unsigned)n);
  DDN_LAUNCH(pack_all_kernel, grid, 256, 0, st, params, cache, t, fp_new, fp_old, force, precision == DDN_PRECISION_BF16X3 ? 1 : 0);
  DDN_LAUNCH(commit_fingerprint_kernel, 1, 32, 0, st, fp_new, fp_old);
  return 0;
}

// ---- fp32-tensor wrappers (single-operator C ABI): split into the staging region, then run the plane kernels
// staging layout: [weights hi|lo][x hi|lo][dy hi|lo][zero-inserted dy hi|lo (stride 2 only)]
size_t tc_workspace_bytes(size_t max_act_elems) { return tc_weight_ws_bytes() + 6 * align_up(max_act_elems * 2, 1024) + 4096; }

static int stage_planes(void* ws, size_t ws_bytes, size_t x_el, size_t dy_el, size_t up_el, void** wws, TcPlanes* x, TcPlanes* dy,
                        TcPlanes* up) {
  char* base = reinterpret_cast<char*>(align_up(reinterpret_cast<uintptr_t>(ws), 1024));
  const size_t wb = align_up(tc_weight_ws_bytes(), 1024), xb = align_up(x_el * 2, 1024), yb = align_up(dy_el * 2, 1024),
               ub = align_up(up_el * 2, 1024);
  if ((size_t)(base - (char*)ws) + wb + 2 * xb + 2 * yb + 2 * ub > ws_bytes) { set_error("tcgen05 staging workspace too small"); return DDN_EWORKSPACE; }
  *wws = base;
  char* q = base + wb;
  x->hi = (__nv_bfloat16*)q; x->lo = (__nv_bfloat16*)(q + xb);
  dy->hi = (__nv_bfloat16*)(q + 2 * xb); dy->lo = (__nv_bfloat16*)(q + 2 * xb + yb);
  up->hi = (__nv_bfloat16*)(q + 2 * xb + 2 * yb); up->lo = (__nv_bfloat16*)(q + 2 * xb + 2 * yb + ub);
  return 0;
}

int tc_conv_forward(const float* x, const float* w, float* y, int N, int H, int W, int Cin, int Cout, int k, int stride, int pad, int dil,
                    int precision, void* ws, size_t ws_bytes, cudaStream_t st) {
  (void)pad;
  void* wws; TcPlanes px, pdy, pup;
  DDN_TRY(stage_planes(ws, ws_bytes, (size_t)N * H * W * Cin, 0, 0, &wws, &px, &pdy, &pup));
  DDN_TRY(tc_split(x, const_cast<__nv_bfloat16*>(px.hi), const_cast<__nv_bfloat16*>(px.lo), (int64_t)N * H * W * Cin, precision, st));
  return tc_conv_planes(px, w, nullptr, y, nullptr, nullptr, N, H, W, Cin, Cout, k, stride, dil, 0, precision, wws, tc_weight_ws_bytes(), st);
}

int tc_conv_backward(const float* x, const float* w, const float* dy, float* dx, const float* dx_addend, float* dw,
                     int N, int H, int W, int Cin, int Cout, int k, int stride, int pad, int dil, int precision,
                     void* ws, size_t ws_bytes, float* dwp_scratch, cudaStream_t st) {
  (void)pad;
  const int Ho = H / stride, Wo = W / stride;
  void* wws; TcPlanes px, pdy, pup;
  DDN_TRY(stage_planes(ws, ws_bytes, (size_t)N * H * W * Cin, (size_t)N * Ho * Wo * Cout, stride == 2 ? (size_t)N * H * W * Cout : 0,
                       &wws, &px, &pdy, &pup));
  DDN_TRY(tc_split(x, const_cast<__nv_bfloat16*>(px.hi), const_cast<__nv_bfloat16*>(px.lo), (int64_t)N * H * W * Cin, precision, st));
  DDN_TRY(tc_split(dy, const_cast<__nv_bfloat16*>(pdy.hi), const_cast<__nv_bfloat16*>(pdy.lo), (int64_t)N * Ho * Wo * Cout, precision, st));
  DDN_TRY(tc_wgrad_planes(px, pdy, dw, N, H, W, Cin, Cout, k, stride, dil, precision, dwp_scratch, st));
  if (dx) {
    if (stride == 2)
      DDN_TRY(tc_dgrad_strided(dy, pup, w, nullptr, dx, dx_addend, N, H, W, Cin, Cout, k, precision, wws, tc_weight_ws_bytes(), st));
    else
      DDN_TRY(tc_conv_planes(pdy, w, nullptr, dx, dx_addend, nullptr, N, H, W, Cin, Cout, k, 1, dil, 1, precision, wws, tc_weight_ws_bytes(), st));
  }
  return 0;
}

}  // namespace ddn
