// Audio front-end kernels of audio2vid: the parts of the wav2vec2-base encoder (transformers Wav2Vec2Model, wrapped by
// reference src/audio_models/wav2vec2.py:13-125) that the GEMM / attention / LayerNorm kernels do not cover.
//
//   wav_conv0_*        feature-extractor layer 0: Conv1d(1, 512, 10, stride 5) + GroupNorm(512, 512) + GELU, three passes
//                      (per-block partial sums -> per-channel affine in double -> recompute the conv, normalise, GELU)
//   interp_time        F.interpolate(linear, align_corners=True) along time (reference torch_utils.py:17-20)
//   pos_conv_gelu      grouped positional convolution (16 groups x 48 channels, k = 128, pad 64, last frame dropped),
//                      GELU and the encoder's residual add, as a tensor-core implicit GEMM per (group, 16-frame tile)
//   mean_f16           fp32 mean over a stack of fp16 matrices (the 13-hidden-state average of model.py:63-66)
#include <mma.h>

#include "ap_host.h"
#include "ap_ptx.cuh"

namespace ap {

__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }

// ---------------------------------------------------------------------------------------------------------
// Layer 0. Block = 512 threads = 512 output channels, CONV0_ROWS output frames; a thread keeps its channel's 10 taps in
// registers and reads the block's waveform segment from shared memory (every thread of a warp reads the same sample:
// broadcast). The conv output is recomputed in the apply pass instead of being stored in fp32 (10 FMAs per value).
// ---------------------------------------------------------------------------------------------------------
constexpr int CONV0_C = 512;
constexpr int CONV0_K = 10;
constexpr int CONV0_S = 5;
constexpr int CONV0_ROWS = 64;
constexpr int CONV0_SEG = (CONV0_ROWS - 1) * CONV0_S + CONV0_K;

__device__ __forceinline__ void conv0_load(const float* __restrict__ wav, long long S, long long r0, float* seg) {
  for (int i = threadIdx.x; i < CONV0_SEG; i += blockDim.x) {
    const long long sidx = r0 * CONV0_S + i;
    seg[i] = sidx < S ? wav[sidx] : 0.f;
  }
}

__device__ __forceinline__ float conv0_at(const float* seg, int r, const float (&w)[CONV0_K]) {
  float v = 0.f;
#pragma unroll
  for (int k = 0; k < CONV0_K; ++k) v = fmaf(w[k], seg[r * CONV0_S + k], v);
  return v;
}

__global__ void __launch_bounds__(CONV0_C)
wav_conv0_stats_kernel(const float* __restrict__ wav, long long S, long long T0, const float* __restrict__ w,
                       float2* __restrict__ partial) {
  griddep_launch_dependents();
  __shared__ float seg[CONV0_SEG];
  const int c = threadIdx.x;
  float wr[CONV0_K];
#pragma unroll
  for (int k = 0; k < CONV0_K; ++k) wr[k] = w[c * CONV0_K + k];
  griddep_wait();
  const long long r0 = (long long)blockIdx.x * CONV0_ROWS;
  conv0_load(wav, S, r0, seg);
  __syncthreads();
  const int rows = (int)min((long long)CONV0_ROWS, T0 - r0);
  float s = 0.f, q = 0.f;
  for (int r = 0; r < rows; ++r) {
    const float v = conv0_at(seg, r, wr);
    s += v;
    q = fmaf(v, v, q);
  }
  partial[(long long)blockIdx.x * CONV0_C + c] = make_float2(s, q);
}

__global__ void __launch_bounds__(CONV0_C)
wav_conv0_finalize_kernel(const float2* __restrict__ partial, int blocks, long long T0, const float* __restrict__ gamma,
                          const float* __restrict__ beta, float eps, float2* __restrict__ affine) {
  griddep_launch_dependents();
  griddep_wait();
  const int c = threadIdx.x;
  double s = 0.0, q = 0.0;
  for (int b = 0; b < blocks; ++b) {   // fixed order: bit-reproducible
    const float2 p = partial[(long long)b * CONV0_C + c];
    s += p.x;
    q += p.y;
  }
  const double mean = s / (double)T0;
  double var = q / (double)T0 - mean * mean;
  var = var > 0.0 ? var : 0.0;
  const double a = (double)gamma[c] / sqrt(var + (double)eps);
  affine[c] = make_float2((float)a, (float)((double)beta[c] - mean * a));
}

__global__ void __launch_bounds__(CONV0_C)
wav_conv0_apply_kernel(const float* __restrict__ wav, long long S, long long T0, const float* __restrict__ w,
                       const float2* __restrict__ affine, __half* __restrict__ out) {
  griddep_launch_dependents();
  __shared__ float seg[CONV0_SEG];
  const int c = threadIdx.x;
  float wr[CONV0_K];
#pragma unroll
  for (int k = 0; k < CONV0_K; ++k) wr[k] = w[c * CONV0_K + k];
  griddep_wait();
  const float2 ab = affine[c];
  const long long r0 = (long long)blockIdx.x * CONV0_ROWS;
  conv0_load(wav, S, r0, seg);
  __syncthreads();
  const int rows = (int)min((long long)CONV0_ROWS, T0 - r0);
  for (int r = 0; r < rows; ++r) {
    const float v = fmaf(conv0_at(seg, r, wr), ab.x, ab.y);
    out[(r0 + r) * CONV0_C + c] = __float2half_rn(gelu_exact(v));
  }
}

// ---------------------------------------------------------------------------------------------------------
// Linear interpolation along time, align_corners=True. Thread = 8 channels of one output frame.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
interp_time_kernel(const __half* __restrict__ x, int T_in, int C, float scale, __half* __restrict__ out, int T_out) {
  griddep_launch_dependents();
  griddep_wait();
  const int cv = C / 8;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)T_out * cv) return;
  const int t = (int)(idx / cv), c8 = (int)(idx % cv) * 8;
  // torch upsample_linear1d (align_corners): src = scale * t, i0 = (int)src, i1 = i0 + (i0 < T_in - 1), l1 = src - i0
  const float src = scale * (float)t;
  int i0 = (int)src;
  if (i0 > T_in - 1) i0 = T_in - 1;
  const int i1 = i0 + (i0 < T_in - 1 ? 1 : 0);
  const float l1 = src - (float)i0, l0 = 1.f - l1;
  const uint4 a = *reinterpret_cast<const uint4*>(x + (long long)i0 * C + c8);
  const uint4 b = *reinterpret_cast<const uint4*>(x + (long long)i1 * C + c8);
  const __half2* ha = reinterpret_cast<const __half2*>(&a);
  const __half2* hb = reinterpret_cast<const __half2*>(&b);
  __half2 o[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 fa = __half22float2(ha[j]), fb = __half22float2(hb[j]);
    o[j] = __floats2half2_rn(l0 * fa.x + l1 * fb.x, l0 * fa.y + l1 * fb.y);
  }
  *reinterpret_cast<uint4*>(out + (long long)t * C + c8) = *reinterpret_cast<const uint4*>(o);
}

// ---------------------------------------------------------------------------------------------------------
// Positional convolution. Block = (16-frame tile, group), 4 warps; warp w takes taps k = 4 j + w (j = 0..31), so the four
// warps share the staged input window and each weight stage (4 taps x 48 x 48) is consumed by all of them. Per tap and warp:
// a [16 frames x 48 in] x [48 in x 48 out] product = 3 x 3 WMMA m16n16k16 steps. The four per-warp accumulators are added in
// warp order at the end (fixed order: bit-reproducible). The input window [t0 - 64, t0 + 16 + 63) with zeros outside [0, T)
// is the conv's zero padding; output frame t < T uses inputs t - 64 .. t + 63 (the SamePad-dropped frame T is never formed).
// ---------------------------------------------------------------------------------------------------------
constexpr int PC_CH = 48;
constexpr int PC_GROUPS = 16;
constexpr int PC_K = 128;
constexpr int PC_PAD = 64;
constexpr int PC_TILE = 16;
constexpr int PC_WIN = PC_TILE + PC_K;          // 144 rows (the last one only pads the window to whole 16-row fragments)
constexpr int PC_STAGE_TAPS = 4;
constexpr int PC_C = PC_CH * PC_GROUPS;         // 768

__global__ void __launch_bounds__(128)
pos_conv_gelu_kernel(const __half* __restrict__ x, int T, const __half* __restrict__ w, const float* __restrict__ bias,
                     __half* __restrict__ out) {
  using namespace nvcuda;
  griddep_launch_dependents();
  __shared__ __align__(128) __half xs[PC_WIN * PC_CH];
  __shared__ __align__(128) __half ws[PC_STAGE_TAPS * PC_CH * PC_CH];
  __shared__ __align__(128) float red[4 * PC_TILE * PC_CH];
  const int warp = threadIdx.x >> 5;
  const int t0 = blockIdx.x * PC_TILE;
  const int g = blockIdx.y;
  const __half* wg = w + (long long)g * PC_K * PC_CH * PC_CH;
  griddep_wait();
  // input window: 144 rows x 48 channels = 6 uint4 per row
  for (int i = threadIdx.x; i < PC_WIN * 6; i += blockDim.x) {
    const int r = i / 6, q = i % 6;
    const int t = t0 - PC_PAD + r;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (t >= 0 && t < T) v = *reinterpret_cast<const uint4*>(x + (long long)t * PC_C + g * PC_CH + q * 8);
    *reinterpret_cast<uint4*>(xs + r * PC_CH + q * 8) = v;
  }
  wmma::fragment<wmma::accumulator, 16, 16, 16, float> acc[3];
#pragma unroll
  for (int o = 0; o < 3; ++o) wmma::fill_fragment(acc[o], 0.f);
  constexpr int STAGE_VEC = PC_STAGE_TAPS * PC_CH * PC_CH / 8;
  for (int k0 = 0; k0 < PC_K; k0 += PC_STAGE_TAPS) {
    __syncthreads();   // previous stage consumed (and, the first time, the window is not yet needed)
    const uint4* src = reinterpret_cast<const uint4*>(wg + (long long)k0 * PC_CH * PC_CH);
    for (int i = threadIdx.x; i < STAGE_VEC; i += blockDim.x) reinterpret_cast<uint4*>(ws)[i] = __ldg(src + i);
    __syncthreads();
    const int k = k0 + warp;
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) {
      wmma::fragment<wmma::matrix_a, 16, 16, 16, __half, wmma::row_major> a;
      wmma::load_matrix_sync(a, xs + k * PC_CH + cc * 16, PC_CH);
#pragma unroll
      for (int o = 0; o < 3; ++o) {
        wmma::fragment<wmma::matrix_b, 16, 16, 16, __half, wmma::row_major> b;
        wmma::load_matrix_sync(b, ws + (warp * PC_CH + cc * 16) * PC_CH + o * 16, PC_CH);
        wmma::mma_sync(acc[o], a, b, acc[o]);
      }
    }
  }
#pragma unroll
  for (int o = 0; o < 3; ++o)
    wmma::store_matrix_sync(red + warp * PC_TILE * PC_CH + o * 16, acc[o], PC_CH, wmma::mem_row_major);
  __syncthreads();
  for (int i = threadIdx.x; i < PC_TILE * PC_CH; i += blockDim.x) {
    const int r = i / PC_CH, o = i % PC_CH;
    const int t = t0 + r;
    if (t >= T) continue;
    const float v = ((red[i] + red[PC_TILE * PC_CH + i]) + red[2 * PC_TILE * PC_CH + i]) + red[3 * PC_TILE * PC_CH + i];
    const int ch = g * PC_CH + o;
    const float res = __half2float(xs[(r + PC_PAD) * PC_CH + o]);
    out[(long long)t * PC_C + ch] = __float2half_rn(res + gelu_exact(v + bias[ch]));
  }
}

// ---------------------------------------------------------------------------------------------------------
// Mean of a stack of fp16 matrices, fp32 sums in source order.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
mean_f16_kernel(const __half* __restrict__ x, int n_src, long long n, float* __restrict__ out_f32,
                __half* __restrict__ out_f16) {
  griddep_launch_dependents();
  griddep_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int k = 0; k < n_src; ++k) s += __half2float(x[(long long)k * n + i]);
  const float m = n_src == 1 ? s : s / (float)n_src;
  if (out_f32) out_f32[i] = m;
  if (out_f16) out_f16[i] = __float2half_rn(m);
}

static long long conv0_frames(long long S) { return S >= CONV0_K ? (S - CONV0_K) / CONV0_S + 1 : 0; }

}  // namespace ap

using namespace ap;

extern "C" int ap_wav_conv0_workspace_floats(long long S) {
  const long long blocks = (conv0_frames(S) + CONV0_ROWS - 1) / CONV0_ROWS;
  const long long floats = 2LL * CONV0_C * (blocks + 1);
  if (floats > 0x7fffffffLL) return fail(AP_ERR_INVALID, "wav_conv0: waveform of %lld samples too long", S);
  return (int)floats;
}

extern "C" int ap_wav_conv0_gn_gelu_f16(const float* wav, long long S, const float* w, const float* gamma,
                                        const float* beta, float eps, float* workspace, long long workspace_floats,
                                        void* out, void* stream) {
  AP_REQUIRE(wav && w && gamma && beta && workspace && out, "wav_conv0: null pointer");
  AP_REQUIRE(S >= CONV0_K, "wav_conv0: %lld samples, fewer than the kernel width %d", S, CONV0_K);
  const long long T0 = conv0_frames(S);
  const long long blocks = (T0 + CONV0_ROWS - 1) / CONV0_ROWS;
  const int need = ap_wav_conv0_workspace_floats(S);
  if (need < 0) return need;
  AP_REQUIRE(workspace_floats >= need, "wav_conv0: workspace of %lld floats, %lld needed",
             workspace_floats, (long long)need);
  float2* partial = reinterpret_cast<float2*>(workspace);
  float2* affine = partial + blocks * CONV0_C;
  AP_LAUNCH(wav_conv0_stats_kernel, (unsigned)blocks, CONV0_C, 0, stream, wav, S, T0, w, partial);
  AP_LAUNCH(wav_conv0_finalize_kernel, 1, CONV0_C, 0, stream, (const float2*)partial, (int)blocks, T0, gamma, beta, eps,
            affine);
  AP_LAUNCH(wav_conv0_apply_kernel, (unsigned)blocks, CONV0_C, 0, stream, wav, S, T0, w, (const float2*)affine,
            (__half*)out);
  AP_CHECK_CUDA(cudaGetLastError());
  return AP_OK;
}

extern "C" int ap_interp_linear_time_f16(const void* x, int T_in, int C, void* out, int T_out, void* stream) {
  AP_REQUIRE(x && out, "interp_linear_time: null pointer");
  AP_REQUIRE(T_in > 0 && T_out > 0 && C > 0 && C % 8 == 0, "interp_linear_time: bad shape T_in=%d T_out=%d C=%d", T_in,
             T_out, C);
  AP_REQUIRE(x != out, "interp_linear_time: out must not alias x");
  const float scale = T_out > 1 ? (float)(T_in - 1) / (float)(T_out - 1) : 0.f;
  const long long n = (long long)T_out * (C / 8);
  AP_LAUNCH(interp_time_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, (const __half*)x, T_in, C, scale,
            (__half*)out, T_out);
  AP_CHECK_CUDA(cudaGetLastError());
  return AP_OK;
}

extern "C" int ap_pos_conv_gelu_f16(const void* x, int T, const void* w, const float* bias, void* out, void* stream) {
  AP_REQUIRE(x && w && bias && out, "pos_conv_gelu: null pointer");
  AP_REQUIRE(T > 0, "pos_conv_gelu: T=%d", T);
  AP_REQUIRE(x != out, "pos_conv_gelu: out must not alias x");
  AP_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0,
             "pos_conv_gelu: x and w must be 16-byte aligned");
  AP_LAUNCH(pos_conv_gelu_kernel, dim3((T + PC_TILE - 1) / PC_TILE, PC_GROUPS), 128, 0, stream, (const __half*)x, T,
            (const __half*)w, bias, (__half*)out);
  AP_CHECK_CUDA(cudaGetLastError());
  return AP_OK;
}

extern "C" int ap_mean_f16(const void* x, int n_src, long long n, float* out_f32, void* out_f16, void* stream) {
  AP_REQUIRE(x && (out_f32 || out_f16), "mean_f16: null pointer");
  AP_REQUIRE(n_src > 0 && n > 0, "mean_f16: bad shape n_src=%d n=%lld", n_src, n);
  AP_LAUNCH(mean_f16_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, (const __half*)x, n_src, n, out_f32,
            (__half*)out_f16);
  AP_CHECK_CUDA(cudaGetLastError());
  return AP_OK;
}
