// Pixelwise contrastive loss fused with the 8x bilinear upsample that precedes it.
//
// The reference evaluates the loss on the full-resolution descriptor image y = upsample_bilinear(low) (resnet_dilated.py:320,
// pixelwise_contrastive_loss.py:131-213): a few thousand descriptors are gathered out of 1.23*D MB per image, and autograd
// scatters their gradients into a zero-filled tensor of that size which the upsample backward then reads in full.  A descriptor
// at pixel (u, v) is a fixed bilinear blend of 4 cells of the LOW-resolution map (60 x 80 x D per image, NHWC here: a cell's D
// channels are one contiguous 4*D-byte row), and that map -- 0.3*D MB for a batch of 16 -- lives in L2.  So these kernels
//   forward : read the two indices of a pair from HBM, 2 x 4 low-resolution cells from L2, blend (the same fp32 arithmetic as
//             upsample_fwd_kernel), squared distance / hinge / count / reduce -- the full-resolution image is never touched;
//   backward: scatter coef * d(l_j)/d(descriptor) * blend weights straight into d(low) (vector reds into an L2-resident
//             array), runs of equal A indices folded by a segmented warp reduction first -- no zero-filled full-resolution
//             gradient, no pass of the upsample backward over it.
// HBM traffic per index pair drops from 16 + 8*D algorithmic bytes (and 8 + 64*D bytes of 32-byte sectors actually moved by
// the channel-strided NCHW gather) to the 16 bytes of the two indices.
//
// Descriptor images: low_a / low_b [B, h*w, D] fp32 (what ddn_resnet34_8s_forward writes to `low_nhwc_out`).
#include <cstdlib>
#include "loss.cuh"

namespace ddn {

constexpr int LR_THREADS = 128;      // small CTAs: the kernels are a single L2 round trip per pair; balance beats reuse

// bilinear source cell + weights of output pixel (u, v): identical arithmetic to head.cu::src_index / upsample_fwd_kernel
struct Blend { int c00, c01, c10, c11; float lh, lw; };
__device__ __forceinline__ Blend blend_of(int64_t n, int W, int h, int w, float sh, float sw) {
  // 0 <= n < H * W < 2^31 (checked by the callers): a 32-bit division -- the 64-bit one is ~80 instructions, and these kernels are
  // instruction-bound (ncu: issue slots 45 % / 65 % busy at C3, DRAM 7 % / 10 %)
  const unsigned ni = (unsigned)n;
  const int v = (int)(ni / (unsigned)W), u = (int)(ni - (unsigned)v * (unsigned)W);
  float r = sh * (float)v;
  int h0 = (int)r; if (h0 > h - 1) h0 = h - 1;
  const int h1 = h0 + ((h0 < h - 1) ? 1 : 0);
  Blend b;
  b.lh = r - (float)h0;
  r = sw * (float)u;
  int w0 = (int)r; if (w0 > w - 1) w0 = w - 1;
  const int w1 = w0 + ((w0 < w - 1) ? 1 : 0);
  b.lw = r - (float)w0;
  b.c00 = h0 * w + w0; b.c01 = h0 * w + w1; b.c10 = h1 * w + w0; b.c11 = h1 * w + w1;
  return b;
}
__device__ __forceinline__ float blend1(float x00, float x01, float x10, float x11, float lh, float lw) {
  const float top = (1.f - lw) * x00 + lw * x01;
  const float bot = (1.f - lw) * x10 + lw * x11;
  return (1.f - lh) * top + lh * bot;
}

// descriptor difference a - b of one pair into d[0..D): D_T > 0 = compile-time D (all 8 * D/4 vector loads are independent and
// issued back to back: one L2 round trip per pair instead of D/4), D_T = 0 = run-time D (scalar loads, any D <= 32)
template <int D_T>
__device__ __forceinline__ void descriptor_diff(const float* __restrict__ A, const float* __restrict__ Bq, const Blend& ba, const Blend& bb,
                                                int D_rt, float (&d)[D_T > 0 ? D_T : LOSS_MAXD]) {
  constexpr int DM = D_T > 0 ? D_T : LOSS_MAXD;
  const int D = D_T > 0 ? D_T : D_rt;
  const float* a00 = A + (size_t)ba.c00 * D; const float* a01 = A + (size_t)ba.c01 * D;
  const float* a10 = A + (size_t)ba.c10 * D; const float* a11 = A + (size_t)ba.c11 * D;
  const float* b00 = Bq + (size_t)bb.c00 * D; const float* b01 = Bq + (size_t)bb.c01 * D;
  const float* b10 = Bq + (size_t)bb.c10 * D; const float* b11 = Bq + (size_t)bb.c11 * D;
  if (D_T > 0 && D_T % 4 == 0) {
    float4 va[D_T / 4 > 0 ? D_T / 4 : 1][4], vb[D_T / 4 > 0 ? D_T / 4 : 1][4];
#pragma unroll
    for (int q = 0; q < D_T / 4; ++q) {
      va[q][0] = __ldg(reinterpret_cast<const float4*>(a00) + q); va[q][1] = __ldg(reinterpret_cast<const float4*>(a01) + q);
      va[q][2] = __ldg(reinterpret_cast<const float4*>(a10) + q); va[q][3] = __ldg(reinterpret_cast<const float4*>(a11) + q);
      vb[q][0] = __ldg(reinterpret_cast<const float4*>(b00) + q); vb[q][1] = __ldg(reinterpret_cast<const float4*>(b01) + q);
      vb[q][2] = __ldg(reinterpret_cast<const float4*>(b10) + q); vb[q][3] = __ldg(reinterpret_cast<const float4*>(b11) + q);
    }
#pragma unroll
    for (int q = 0; q < D_T / 4; ++q) {
      d[4 * q + 0] = blend1(va[q][0].x, va[q][1].x, va[q][2].x, va[q][3].x, ba.lh, ba.lw) - blend1(vb[q][0].x, vb[q][1].x, vb[q][2].x, vb[q][3].x, bb.lh, bb.lw);
      d[4 * q + 1] = blend1(va[q][0].y, va[q][1].y, va[q][2].y, va[q][3].y, ba.lh, ba.lw) - blend1(vb[q][0].y, vb[q][1].y, vb[q][2].y, vb[q][3].y, bb.lh, bb.lw);
      d[4 * q + 2] = blend1(va[q][0].z, va[q][1].z, va[q][2].z, va[q][3].z, ba.lh, ba.lw) - blend1(vb[q][0].z, vb[q][1].z, vb[q][2].z, vb[q][3].z, bb.lh, bb.lw);
      d[4 * q + 3] = blend1(va[q][0].w, va[q][1].w, va[q][2].w, va[q][3].w, ba.lh, ba.lw) - blend1(vb[q][0].w, vb[q][1].w, vb[q][2].w, vb[q][3].w, bb.lh, bb.lw);
    }
  } else {
#pragma unroll
    for (int c = 0; c < DM; ++c) {
      d[c] = 0.f;
      if (c < D)
        d[c] = blend1(__ldg(a00 + c), __ldg(a01 + c), __ldg(a10 + c), __ldg(a11 + c), ba.lh, ba.lw) -
               blend1(__ldg(b00 + c), __ldg(b01 + c), __ldg(b10 + c), __ldg(b11 + c), bb.lh, bb.lw);
    }
  }
}

template <int D_T>
__global__ void __launch_bounds__(LR_THREADS)
loss_lowres_fwd_kernel(const float* __restrict__ la, const float* __restrict__ lb, int h, int w, int H, int W, int D_rt, float sh, float sw,
                       const __grid_constant__ DevTerms T, double* __restrict__ sums, unsigned long long* __restrict__ counts) {
  pdl_prologue();
  constexpr int DM = D_T > 0 ? D_T : LOSS_MAXD;
  const int D = D_T > 0 ? D_T : D_rt;
  const int b = blockIdx.y;
  const int t = find_term(T, blockIdx.x);
  const DevTerm& tm = T.t[t];
  const int64_t P = (int64_t)H * W;
  const int64_t cells = (int64_t)h * w;
  const float* A = la + (size_t)b * cells * D;
  const float* Bq = lb + (size_t)b * cells * D;
  const int64_t nvalid = tm.len ? min(tm.len[b], tm.n) : tm.n;
  const int64_t j = (int64_t)(blockIdx.x - tm.block_begin) * LR_THREADS + threadIdx.x;
  float acc = 0.f;
  int cnt = 0;
  if (j < nvalid) {
    const int64_t na = __ldg(tm.ia + b * tm.n + j), nb = __ldg(tm.ib + b * tm.n + j);
    if (na >= 0 && nb >= 0 && na < P && nb < P) {
      const Blend ba = blend_of(na, W, h, w, sh, sw), bb = blend_of(nb, W, h, w, sh, sw);
      float d[DM];
      descriptor_diff<D_T>(A, Bq, ba, bb, D, d);
      float s2 = 0.f;
#pragma unroll
      for (int c = 0; c < DM; ++c) s2 = fmaf(d[c], d[c], s2);
      if (tm.kind == DDN_TERM_MATCH) {
        acc = s2;
      } else {
        const float dist = sqrtf(s2);
        const float hg = (tm.kind == DDN_TERM_HINGE) ? fmaxf(tm.margin - dist, 0.f) : fmaxf(dist - tm.margin, 0.f);
        float l = hg * hg;
        cnt = (l != 0.f);
        if (tm.flags & DDN_TERM_PIXEL_WEIGHT) l *= pixel_weight(tm, b, j, nb, W);
        acc = l;
      }
    }
  }
  double wsum = warp_sum((double)acc);
  int wcnt = warp_sum(cnt);
  __shared__ double s_sum[LR_THREADS / 32];
  __shared__ int s_cnt[LR_THREADS / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { s_sum[wid] = wsum; s_cnt[wid] = wcnt; }
  __syncthreads();
  if (wid == 0) {
    double v = lane < LR_THREADS / 32 ? s_sum[lane] : 0.0;
    int c = lane < LR_THREADS / 32 ? s_cnt[lane] : 0;
    v = warp_sum(v);
    c = warp_sum(c);
    if (lane == 0) {
      if (v != 0.0) atomicAdd(&sums[b * T.n_terms + t], v);
      if (c) atomicAdd(&counts[b * T.n_terms + t], (unsigned long long)c);
    }
  }
}

__device__ __forceinline__ void red_add_v4f(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// scatter g[0..D) * blend weights into the 4 cells of pixel `bl` (vector reds when D is a multiple of 4)
template <int D_T>
__device__ __forceinline__ void scatter_desc(float* __restrict__ dL, const Blend& bl, int D_rt, const float (&g)[D_T > 0 ? D_T : LOSS_MAXD]) {
  constexpr int DM = D_T > 0 ? D_T : LOSS_MAXD;
  const int D = D_T > 0 ? D_T : D_rt;
  const float wts[4] = {(1.f - bl.lh) * (1.f - bl.lw), (1.f - bl.lh) * bl.lw, bl.lh * (1.f - bl.lw), bl.lh * bl.lw};
  const int cell[4] = {bl.c00, bl.c01, bl.c10, bl.c11};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float wk = wts[k];
    if (k > 0 && wk == 0.f) continue;           // clamped edge cells coincide with cell 0 and carry weight 0
    float* dst = dL + (size_t)cell[k] * D;
    if (D_T > 0 && D_T % 4 == 0) {
#pragma unroll
      for (int q = 0; q < DM / 4; ++q) red_add_v4f(dst + 4 * q, wk * g[4 * q], wk * g[4 * q + 1], wk * g[4 * q + 2], wk * g[4 * q + 3]);
    } else {
#pragma unroll
      for (int c = 0; c < DM; ++c)
        if (c < D) atomicAdd(dst + c, wk * g[c]);
    }
  }
}

template <int D_T>
__global__ void __launch_bounds__(LR_THREADS)
loss_lowres_bwd_kernel(const float* __restrict__ la, const float* __restrict__ lb, int h, int w, int H, int W, int D_rt, float sh, float sw,
                       const __grid_constant__ DevTerms T, const float* __restrict__ coef, const float* __restrict__ upstream,
                       float* __restrict__ dla, float* __restrict__ dlb) {
  pdl_prologue();
  constexpr int DM = D_T > 0 ? D_T : LOSS_MAXD;
  const int D = D_T > 0 ? D_T : D_rt;
  const int b = blockIdx.y;
  const int t = find_term(T, blockIdx.x);
  const DevTerm& tm = T.t[t];
  float cf = coef[b * T.n_terms + t];
  if (upstream) cf *= upstream[0];
  const int64_t P = (int64_t)H * W;
  const int64_t cells = (int64_t)h * w;
  const float* A = la + (size_t)b * cells * D;
  const float* Bq = lb + (size_t)b * cells * D;
  float* dA = dla + (size_t)b * cells * D;
  float* dB = dlb + (size_t)b * cells * D;
  const int64_t nvalid = tm.len ? min(tm.len[b], tm.n) : tm.n;
  const int64_t j = (int64_t)(blockIdx.x - tm.block_begin) * LR_THREADS + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool hinge = tm.kind != DDN_TERM_MATCH;
  int64_t na = -1, nb = -1;
  if (j < nvalid) { na = __ldg(tm.ia + b * tm.n + j); nb = __ldg(tm.ib + b * tm.n + j); }
  const bool ok = na >= 0 && nb >= 0 && na < P && nb < P;
  Blend ba = {}, bb = {};
  float g[DM];
#pragma unroll
  for (int c = 0; c < DM; ++c) g[c] = 0.f;
  float scale = 0.f;
  if (ok) {
    ba = blend_of(na, W, h, w, sh, sw); bb = blend_of(nb, W, h, w, sh, sw);
    descriptor_diff<D_T>(A, Bq, ba, bb, D, g);
    float s2 = 0.f;
#pragma unroll
    for (int c = 0; c < DM; ++c) s2 = fmaf(g[c], g[c], s2);
    if (!hinge) {
      scale = 2.f * cf;                                  // d/dA ||A-B||^2
    } else {
      const float dist = sqrtf(s2);
      const float hg = (tm.kind == DDN_TERM_HINGE) ? fmaxf(tm.margin - dist, 0.f) : fmaxf(dist - tm.margin, 0.f);
      if (hg * hg != 0.f && dist > 0.f) {                // norm's subgradient at 0 is 0 (torch)
        const float wgt = (tm.flags & DDN_TERM_PIXEL_WEIGHT) ? pixel_weight(tm, b, j, nb, W) : 1.f;
        const float sgn = (tm.kind == DDN_TERM_HINGE) ? -1.f : 1.f;
        scale = cf * wgt * sgn * 2.f * hg / dist;
      }
    }
  }
#pragma unroll
  for (int c = 0; c < DM; ++c) g[c] *= scale;
  if (ok && scale != 0.f) {                              // B side: random indices
    float gb[DM];
#pragma unroll
    for (int c = 0; c < DM; ++c) gb[c] = -g[c];
    scatter_desc<D_T>(dB, bb, D, gb);
  }
  if (!hinge) {
    if (ok && scale != 0.f) scatter_desc<D_T>(dA, ba, D, g);
    return;
  }
  // runs of equal A indices (every match repeated k times consecutively, spartan_dataset_masked.py:853-854): one scatter per run
  const int64_t key = ok ? na : (int64_t)(-1 - lane);
  const int64_t prev = __shfl_up_sync(0xffffffffu, key, 1);
  const bool head = (lane == 0) || (prev != key);
  const unsigned heads = __ballot_sync(0xffffffffu, head);
  const unsigned above = heads & ~((2u << lane) - 1u);
  const int run_end = above ? (__ffs(above) - 2) : 31;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const bool take = (lane + off) <= run_end;
#pragma unroll
    for (int c = 0; c < DM; ++c) {
      if (c < D) {
        const float o = __shfl_down_sync(0xffffffffu, g[c], off);
        if (take) g[c] += o;
      }
    }
  }
  if (head && ok) {
    bool any = false;
#pragma unroll
    for (int c = 0; c < DM; ++c) any = any || (g[c] != 0.f);
    if (any) scatter_desc<D_T>(dA, ba, D, g);
  }
}

// ---- D = 8 / 16 / 32: LPP = D / 4 lanes per index pair, one channel QUAD per lane.  A warp instruction then touches one 16 * LPP-byte
// piece of a cell per pair instead of one line per LANE (the one-pair-per-lane kernels above spend their time in L1 tag lookups:
// 32 scattered 16-byte loads per instruction), every lane keeps 8 loads in flight instead of 2 * D, and the backward's segmented
// run reduction moves 4 floats per lane per step instead of D.
template <int LPP>
__device__ __forceinline__ float4 quad_diff(const float* __restrict__ A, const float* __restrict__ Bq, const Blend& ba, const Blend& bb, int sub) {
  constexpr int D = 4 * LPP;
  const float4 a00 = __ldg(reinterpret_cast<const float4*>(A + (size_t)ba.c00 * D) + sub), a01 = __ldg(reinterpret_cast<const float4*>(A + (size_t)ba.c01 * D) + sub);
  const float4 a10 = __ldg(reinterpret_cast<const float4*>(A + (size_t)ba.c10 * D) + sub), a11 = __ldg(reinterpret_cast<const float4*>(A + (size_t)ba.c11 * D) + sub);
  const float4 b00 = __ldg(reinterpret_cast<const float4*>(Bq + (size_t)bb.c00 * D) + sub), b01 = __ldg(reinterpret_cast<const float4*>(Bq + (size_t)bb.c01 * D) + sub);
  const float4 b10 = __ldg(reinterpret_cast<const float4*>(Bq + (size_t)bb.c10 * D) + sub), b11 = __ldg(reinterpret_cast<const float4*>(Bq + (size_t)bb.c11 * D) + sub);
  return make_float4(blend1(a00.x, a01.x, a10.x, a11.x, ba.lh, ba.lw) - blend1(b00.x, b01.x, b10.x, b11.x, bb.lh, bb.lw),
                     blend1(a00.y, a01.y, a10.y, a11.y, ba.lh, ba.lw) - blend1(b00.y, b01.y, b10.y, b11.y, bb.lh, bb.lw),
                     blend1(a00.z, a01.z, a10.z, a11.z, ba.lh, ba.lw) - blend1(b00.z, b01.z, b10.z, b11.z, bb.lh, bb.lw),
                     blend1(a00.w, a01.w, a10.w, a11.w, ba.lh, ba.lw) - blend1(b00.w, b01.w, b10.w, b11.w, bb.lh, bb.lw));
}

// LR_FWD_ITEMS index pairs per lane group in the forward: that many times fewer blocks = fewer contended atomics on the
// B * n_terms accumulators (they bound the one-pair version), and 8 * LR_FWD_ITEMS loads in flight per lane
template <int LPP, int LR_FWD_ITEMS>
__global__ void __launch_bounds__(LR_THREADS)
loss_lowres_fwd_quad_kernel(const float* __restrict__ la, const float* __restrict__ lb, int h, int w, int H, int W, float sh, float sw,
                            const __grid_constant__ DevTerms T, double* __restrict__ sums, unsigned long long* __restrict__ counts) {
  pdl_prologue();
  constexpr int D = 4 * LPP, PPB = LR_THREADS / LPP;
  const int b = blockIdx.y;
  const int t = find_term(T, blockIdx.x);
  const DevTerm& tm = T.t[t];
  const int64_t P = (int64_t)H * W;
  const int64_t cells = (int64_t)h * w;
  const float* A = la + (size_t)b * cells * D;
  const float* Bq = lb + (size_t)b * cells * D;
  const int64_t nvalid = tm.len ? min(tm.len[b], tm.n) : tm.n;
  const int sub = threadIdx.x % LPP;
  const int64_t j0 = (int64_t)(blockIdx.x - tm.block_begin) * (PPB * LR_FWD_ITEMS) + threadIdx.x / LPP;
  int64_t na[LR_FWD_ITEMS], nb[LR_FWD_ITEMS];
#pragma unroll
  for (int k = 0; k < LR_FWD_ITEMS; ++k) {
    const int64_t j = j0 + k * PPB;
    na[k] = -1; nb[k] = -1;
    if (j < nvalid) { na[k] = __ldg(tm.ia + b * tm.n + j); nb[k] = __ldg(tm.ib + b * tm.n + j); }
  }
  float s2[LR_FWD_ITEMS];
  bool ok[LR_FWD_ITEMS];
#pragma unroll
  for (int k = 0; k < LR_FWD_ITEMS; ++k) {
    ok[k] = na[k] >= 0 && nb[k] >= 0 && na[k] < P && nb[k] < P;
    s2[k] = 0.f;
    if (ok[k]) {
      const Blend ba = blend_of(na[k], W, h, w, sh, sw), bb = blend_of(nb[k], W, h, w, sh, sw);
      const float4 d = quad_diff<LPP>(A, Bq, ba, bb, sub);
      s2[k] = fmaf(d.x, d.x, fmaf(d.y, d.y, fmaf(d.z, d.z, d.w * d.w)));
    }
  }
  float acc = 0.f;
  int cnt = 0;
#pragma unroll
  for (int k = 0; k < LR_FWD_ITEMS; ++k) {
    float v = s2[k];
#pragma unroll
    for (int off = 1; off < LPP; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (ok[k] && sub == 0) {
      if (tm.kind == DDN_TERM_MATCH) {
        acc += v;
      } else {
        const float dist = sqrtf(v);
        const float hg = (tm.kind == DDN_TERM_HINGE) ? fmaxf(tm.margin - dist, 0.f) : fmaxf(dist - tm.margin, 0.f);
        float l = hg * hg;
        cnt += (l != 0.f);
        if (tm.flags & DDN_TERM_PIXEL_WEIGHT) l *= pixel_weight(tm, b, j0 + k * PPB, nb[k], W);
        acc += l;
      }
    }
  }
  double wsum = warp_sum((double)acc);
  int wcnt = warp_sum(cnt);
  __shared__ double s_sum[LR_THREADS / 32];
  __shared__ int s_cnt[LR_THREADS / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { s_sum[wid] = wsum; s_cnt[wid] = wcnt; }
  __syncthreads();
  if (wid == 0) {
    double v = lane < LR_THREADS / 32 ? s_sum[lane] : 0.0;
    int c = lane < LR_THREADS / 32 ? s_cnt[lane] : 0;
    v = warp_sum(v);
    c = warp_sum(c);
    if (lane == 0) {
      if (v != 0.0) atomicAdd(&sums[b * T.n_terms + t], v);
      if (c) atomicAdd(&counts[b * T.n_terms + t], (unsigned long long)c);
    }
  }
}

template <int LPP>
__device__ __forceinline__ void scatter_quad(float* __restrict__ dL, const Blend& bl, int sub, float4 g) {
  constexpr int D = 4 * LPP;
  const float wts[4] = {(1.f - bl.lh) * (1.f - bl.lw), (1.f - bl.lh) * bl.lw, bl.lh * (1.f - bl.lw), bl.lh * bl.lw};
  const int cell[4] = {bl.c00, bl.c01, bl.c10, bl.c11};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float wk = wts[k];
    if (k > 0 && wk == 0.f) continue;           // clamped edge cells coincide with cell 0 and carry weight 0
    red_add_v4f(dL + (size_t)cell[k] * D + 4 * sub, wk * g.x, wk * g.y, wk * g.z, wk * g.w);
  }
}

template <int LPP>
__global__ void __launch_bounds__(LR_THREADS)
loss_lowres_bwd_quad_kernel(const float* __restrict__ la, const float* __restrict__ lb, int h, int w, int H, int W, float sh, float sw,
                            const __grid_constant__ DevTerms T, const float* __restrict__ coef, const float* __restrict__ upstream,
                            float* __restrict__ dla, float* __restrict__ dlb) {
  pdl_prologue();
  constexpr int D = 4 * LPP, PPB = LR_THREADS / LPP, PPW = 32 / LPP;      // pairs per block / per warp
  const int b = blockIdx.y;
  const int t = find_term(T, blockIdx.x);
  const DevTerm& tm = T.t[t];
  float cf = coef[b * T.n_terms + t];
  if (upstream) cf *= upstream[0];
  const int64_t P = (int64_t)H * W;
  const int64_t cells = (int64_t)h * w;
  const float* A = la + (size_t)b * cells * D;
  const float* Bq = lb + (size_t)b * cells * D;
  float* dA = dla + (size_t)b * cells * D;
  float* dB = dlb + (size_t)b * cells * D;
  const int64_t nvalid = tm.len ? min(tm.len[b], tm.n) : tm.n;
  const int lane = threadIdx.x & 31;
  const int sub = lane % LPP, pidx = lane / LPP;
  const int64_t j = (int64_t)(blockIdx.x - tm.block_begin) * PPB + threadIdx.x / LPP;
  const bool hinge = tm.kind != DDN_TERM_MATCH;
  int64_t na = -1, nb = -1;
  if (j < nvalid) { na = __ldg(tm.ia + b * tm.n + j); nb = __ldg(tm.ib + b * tm.n + j); }
  const bool ok = na >= 0 && nb >= 0 && na < P && nb < P;
  Blend ba = {}, bb = {};
  float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
  float s2 = 0.f;
  if (ok) {
    ba = blend_of(na, W, h, w, sh, sw); bb = blend_of(nb, W, h, w, sh, sw);
    g = quad_diff<LPP>(A, Bq, ba, bb, sub);
    s2 = fmaf(g.x, g.x, fmaf(g.y, g.y, fmaf(g.z, g.z, g.w * g.w)));
  }
#pragma unroll
  for (int off = 1; off < LPP; off <<= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, off);
  float scale = 0.f;
  if (ok) {
    if (!hinge) {
      scale = 2.f * cf;                                  // d/dA ||A-B||^2
    } else {
      const float dist = sqrtf(s2);
      const float hg = (tm.kind == DDN_TERM_HINGE) ? fmaxf(tm.margin - dist, 0.f) : fmaxf(dist - tm.margin, 0.f);
      if (hg * hg != 0.f && dist > 0.f) {                // norm's subgradient at 0 is 0 (torch)
        const float wgt = (tm.flags & DDN_TERM_PIXEL_WEIGHT) ? pixel_weight(tm, b, j, nb, W) : 1.f;
        const float sgn = (tm.kind == DDN_TERM_HINGE) ? -1.f : 1.f;
        scale = cf * wgt * sgn * 2.f * hg / dist;
      }
    }
  }
  g.x *= scale; g.y *= scale; g.z *= scale; g.w *= scale;
  if (ok && scale != 0.f) scatter_quad<LPP>(dB, bb, sub, make_float4(-g.x, -g.y, -g.z, -g.w));       // B side: random indices
  if (!hinge) {
    if (ok && scale != 0.f) scatter_quad<LPP>(dA, ba, sub, g);
    return;
  }
  // runs of equal A indices (every match repeated k times consecutively, spartan_dataset_masked.py:853-854): one scatter per run
  const int64_t key = ok ? na : (int64_t)(-1 - pidx);
  const int64_t prev = __shfl_up_sync(0xffffffffu, key, LPP);
  const bool head = (pidx == 0) || (prev != key);
  const unsigned heads = __ballot_sync(0xffffffffu, head);
  const unsigned below_next = (pidx + 1 == PPW) ? 0xffffffffu : ((1u << ((pidx + 1) * LPP)) - 1u);    // lanes of pairs <= mine
  const unsigned above = heads & ~below_next;
  const int run_end = above ? ((__ffs(above) - 1) / LPP - 1) : (PPW - 1);                               // last pair of my run
#pragma unroll
  for (int off = 1; off < PPW; off <<= 1) {
    const bool take = (pidx + off) <= run_end;
    const float ox = __shfl_down_sync(0xffffffffu, g.x, off * LPP), oy = __shfl_down_sync(0xffffffffu, g.y, off * LPP);
    const float oz = __shfl_down_sync(0xffffffffu, g.z, off * LPP), ow = __shfl_down_sync(0xffffffffu, g.w, off * LPP);
    if (take) { g.x += ox; g.y += oy; g.z += oz; g.w += ow; }
  }
  if (head && ok && (g.x != 0.f || g.y != 0.f || g.z != 0.f || g.w != 0.f)) scatter_quad<LPP>(dA, ba, sub, g);
}

static int build_terms_lr(const ddn_loss_term* th, int n_terms, DevTerms* T, int pairs_per_block = LR_THREADS) {
  DDN_TRY(build_terms(th, n_terms, T));
  int blk = 0;                                   // one index pair per thread (or per D / 4 threads: the quad kernels)
  for (int i = 0; i < n_terms; ++i) { T->t[i].block_begin = blk; blk += (int)ceil_div(th[i].n, pairs_per_block); }
  T->total_blocks = blk;
  return 0;
}
static float ac_scale(int in, int out) { return out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.f; }

// The D = 4 / 8 / 16 / 32 kernels read and reduce 16-byte vectors, so their maps must start 16-byte aligned; a cell row is then a
// multiple of 16 bytes for every D % 4 == 0.  The other D take scalar accesses and accept any float-aligned map -- e.g. the
// second half of forward_pair's output at D = 3, which starts B * h * w * 12 bytes into the buffer.
static bool lowres_aligned(int D, const void* a, const void* b, const void* c = nullptr, const void* d = nullptr) {
  if (D % 4 != 0) return true;
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c) | reinterpret_cast<uintptr_t>(d)) & 15) == 0;
}

}  // namespace ddn

using namespace ddn;

extern "C" int ddn_contrastive_terms_forward_lowres(const float* low_a, const float* low_b, int B, int h, int w, int H, int W, int D,
                                                    const ddn_loss_term* terms_host, int n_terms,
                                                    double* sums, int64_t* counts, void* stream) {
  DDN_TRY(check_common(low_a, low_b, B, (int64_t)H * W, D, W));
  DDN_CHECK_ARG(sums && counts && h >= 1 && w >= 1 && H >= h && W >= w && (int64_t)H * W < (1LL << 31), "bad low-resolution geometry / null outputs");
  DDN_CHECK_ARG(lowres_aligned(D, low_a, low_b), "low-resolution maps must be 16-byte aligned when D is a multiple of 4");
  const int lpp = (D == 8 || D == 16 || D == 32) ? D / 4 : 1;
  // 4 pairs per lane group; 8 halves the atomics again but costs occupancy: 17.4 -> 18.7-20.9 us at C3 (DESIGN.md §8)
  constexpr int items = 4;
  DevTerms T;
  DDN_TRY(build_terms_lr(terms_host, n_terms, &T, lpp > 1 ? LR_THREADS / lpp * items : LR_THREADS));
  cudaStream_t st = (cudaStream_t)stream;
  DDN_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * B * n_terms, st));
  DDN_CUDA(cudaMemsetAsync(counts, 0, sizeof(int64_t) * B * n_terms, st));
  if (T.total_blocks == 0) return 0;
  dim3 grid(T.total_blocks, B);
  auto cnt = reinterpret_cast<unsigned long long*>(counts);
  double pairs = 0;
  for (int i = 0; i < n_terms; ++i) pairs += (double)terms_host[i].n * B;
  ProfScope ps(PROF_LOSS_FWD, pairs * (16.0 + 8.0 * D), st);
  const float sh = ac_scale(h, H), sw = ac_scale(w, W);
#define FWD(DT) DDN_LAUNCH(loss_lowres_fwd_kernel<DT>, grid, LR_THREADS, 0, st, low_a, low_b, h, w, H, W, D, sh, sw, T, sums, cnt)
#define FWDQ(L) DDN_LAUNCH((loss_lowres_fwd_quad_kernel<L, items>), grid, LR_THREADS, 0, st, low_a, low_b, h, w, H, W, sh, sw, T, sums, cnt)
  switch (D) {
    case 3: FWD(3); break;
    case 4: FWD(4); break;
    case 8: FWDQ(2); break;
    case 16: FWDQ(4); break;
    case 32: FWDQ(8); break;
    default: FWD(0); break;
  }
#undef FWD
#undef FWDQ
  return 0;
}

extern "C" int ddn_contrastive_terms_backward_lowres(const float* low_a, const float* low_b, int B, int h, int w, int H, int W, int D,
                                                     const ddn_loss_term* terms_host, int n_terms,
                                                     const float* coef, const float* upstream,
                                                     float* dlow_a, float* dlow_b, void* stream) {
  DDN_TRY(check_common(low_a, low_b, B, (int64_t)H * W, D, W));
  DDN_CHECK_ARG(coef && dlow_a && dlow_b && h >= 1 && w >= 1 && H >= h && W >= w && (int64_t)H * W < (1LL << 31), "bad low-resolution geometry / null buffers");
  DDN_CHECK_ARG(lowres_aligned(D, low_a, low_b, dlow_a, dlow_b),
                "low-resolution maps and their gradients must be 16-byte aligned when D is a multiple of 4");
  const int lpp = (D == 8 || D == 16 || D == 32) ? D / 4 : 1;
  DevTerms T;
  DDN_TRY(build_terms_lr(terms_host, n_terms, &T, LR_THREADS / lpp));
  if (T.total_blocks == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(T.total_blocks, B);
  double pairs = 0;
  for (int i = 0; i < n_terms; ++i) pairs += (double)terms_host[i].n * B;
  ProfScope ps(PROF_LOSS_BWD, pairs * (16.0 + 24.0 * D), st);
  const float sh = ac_scale(h, H), sw = ac_scale(w, W);
#define BWD(DT) DDN_LAUNCH(loss_lowres_bwd_kernel<DT>, grid, LR_THREADS, 0, st, low_a, low_b, h, w, H, W, D, sh, sw, T, coef, upstream, dlow_a, dlow_b)
#define BWDQ(L) DDN_LAUNCH(loss_lowres_bwd_quad_kernel<L>, grid, LR_THREADS, 0, st, low_a, low_b, h, w, H, W, sh, sw, T, coef, upstream, dlow_a, dlow_b)
  switch (D) {
    case 3: BWD(3); break;
    case 4: BWD(4); break;
    case 8: BWDQ(2); break;
    case 16: BWDQ(4); break;
    case 32: BWDQ(8); break;
    default: BWD(0); break;
  }
#undef BWD
#undef BWDQ
  return 0;
}
