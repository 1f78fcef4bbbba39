// tcgen05 (5th-gen tensor core) implicit-GEMM convolution interface -- see conv_tc.cu.
#pragma once
#include "common.cuh"
#include "bn_stats.cuh"

namespace ddn {

struct TcPlanes { const __nv_bfloat16* hi; const __nv_bfloat16* lo; };   // x ~= hi + lo (lo unused in single-pass bf16)

// Inference epilogue of a forward conv: y = relu?(conv * scale[c] + shift[c] + addend) -- BatchNorm in eval mode folded into
// the conv (scale = gamma / sqrt(running_var + eps), shift = beta - running_mean * scale) -- written as fp32 (`out`, may be
// null) and / or as the bf16 hi/lo operand planes of the next conv.
struct TcFoldedEpilogue { const float* scale; const float* shift; int relu; __nv_bfloat16* out_hi; __nv_bfloat16* out_lo; };

// Data-gradient epilogue that also produces the column sums of the BatchNorm backward consuming the gradient it writes:
// out = dY of y = relu?(bn(raw) [+ residual]); g = out * (y > 0) with the mask taken from the bf16 hi plane of y (`y_hi`, blocks
// with a residual) or recomputed from raw (relu, no residual); (sum g, sum g * xhat) per channel and BatchNorm group go through
// fin.a, and the kernel's last CTA writes fin.sums / dgamma / dbeta -- exactly what bn_colsum_kernel<1> would, one pass earlier.
struct TcBwdStats {
  const float* raw; const __nv_bfloat16* y_hi;
  const float* mean; const float* invstd;      // [G][C]
  const float* gamma; const float* beta;       // [C]
  int relu;
  BnBwdFinal fin;
};

bool tc_available();
// forward / weight gradient: 3x3 (pad == dil) or 1x1 (pad 0), Cin and Cout multiples of 64, stride 1 (any dil) or 2 (dil 1)
bool tc_conv_supported(int Cin, int Cout, int k, int stride, int pad, int dil, int H, int W);
size_t tc_weight_ws_bytes();                       // staging for one conv's packed bf16 weights
size_t tc_workspace_bytes(size_t max_act_elems);   // staging for the fp32-tensor wrappers below
int tc_split(const float* x, __nv_bfloat16* hi, __nv_bfloat16* lo, int64_t n, int precision, cudaStream_t st);

// plane-level entry points (what the network engine calls)
// stats != nullptr (forward): the epilogue accumulates the per-channel sum / sum of squares of the output and the kernel's last
// CTA writes the BatchNorm statistics (bn_stats.cuh); stats->G BatchNorm groups of N / G images each.
int tc_conv_planes(TcPlanes in, const float* w_oihw, const TcPlanes* w_packed, float* out, const float* addend, const BnFwdFinal* stats,
                   int N, int H, int W, int Cin, int Cout, int k, int stride, int dil, int dgrad, int precision,
                   void* wws, size_t wws_bytes, cudaStream_t st, const TcFoldedEpilogue* ep = nullptr, const TcBwdStats* bst = nullptr);
int tc_pack_weights(const float* w_oihw, __nv_bfloat16* hi, __nv_bfloat16* lo, int Cout, int Cin, int k, int dgrad, int precision,
                    cudaStream_t st);
int tc_dgrad_strided(const float* dy_f32, TcPlanes up, const float* w_oihw, const TcPlanes* w_packed, float* dx, const float* addend,
                     int N, int H, int W, int Cin, int Cout, int k, int precision, void* wws, size_t wws_bytes, cudaStream_t st,
                     const TcBwdStats* bst = nullptr);
// dw != nullptr: immediate (dwp = scratch, zero-filled and converted here); dw == nullptr: accumulate into the caller's pre-zeroed
// dwp [taps][Cout][Cin] and convert later with tc_unpack_wgrads (one launch for a whole gradient bucket)
int tc_wgrad_planes(TcPlanes x, TcPlanes dy, float* dw, int N, int H, int W, int Cin, int Cout, int k, int stride, int dil,
                    int precision, float* dwp, cudaStream_t st);
struct TcUnpackEntry { int64_t src_off, dst_off; int Cout, Cin, taps, kind; };   // kind 1 = stem [64][192] -> [64][3][7][7]
constexpr int TC_UNPACK_MAX = 40;
struct TcUnpackTable { TcUnpackEntry e[TC_UNPACK_MAX]; int n; };
int tc_unpack_wgrads(const TcUnpackEntry* entries, int n, const float* dwp_base, float* grads_base, cudaStream_t st);
// device-validated cache of every conv's packed weights (see conv_tc.cu "weight-pack cache")
struct TcPackEntry { int64_t w_off, dst_off; int Cout, Cin, k, dgrad, kind; };   // kind 1 = stem patch-GEMM layout [64][192]
constexpr int TC_PACK_MAX = 80;
struct TcPackTable { TcPackEntry e[TC_PACK_MAX]; int n; };
int tc_pack_all(const float* params, int64_t n_params, char* cache, const TcPackEntry* entries, int n, unsigned long long* fp_new,
                unsigned long long* fp_old, int force, int precision, cudaStream_t st);
// stem conv1 (7x7/2, Cin = 3) as a K = 192 GEMM over patch planes [N,H1,W1,192]
int tc_stem_patches(const float* x_nchw, __nv_bfloat16* hi, __nv_bfloat16* lo, int N, int H, int W, int precision, cudaStream_t st);
int tc_stem_pack_weights(const float* w_conv1, __nv_bfloat16* hi, __nv_bfloat16* lo, int precision, cudaStream_t st);   // [64][192]
int tc_stem_forward(TcPlanes patches, const float* w_conv1, const TcPlanes* w_packed, float* raw, const BnFwdFinal* stats, int N, int H1,
                    int W1, int precision, void* wws, size_t wws_bytes, cudaStream_t st);
int tc_stem_wgrad(TcPlanes patches, TcPlanes dy, float* dw_conv1, int N, int H1, int W1, int precision, float* scratch, cudaStream_t st);

// fp32-tensor wrappers (single-operator C ABI)
int tc_conv_forward(const float* x_nhwc, const float* w_oihw, float* y_nhwc, int N, int H, int W, int Cin, int Cout,
                    int k, int stride, int pad, int dil, int precision, void* ws, size_t ws_bytes, cudaStream_t st);
int tc_conv_backward(const float* x_nhwc, const float* w_oihw, const float* dy_nhwc, float* dx_nhwc, const float* dx_addend,
                     float* dw_oihw, int N, int H, int W, int Cin, int Cout, int k, int stride, int pad, int dil, int precision,
                     void* ws, size_t ws_bytes, float* dwp_scratch, cudaStream_t st);

}  // namespace ddn
