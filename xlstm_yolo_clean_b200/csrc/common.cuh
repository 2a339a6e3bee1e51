// Shared device/host helpers for the sm_100a mLSTM chunkwise kernels.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/mlstm_b200.h"

namespace mlstm {

// ---------------------------------------------------------------------------------------------
// host-side bookkeeping shared by the C-ABI translation units
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define MLSTM_CUDA_CHECK(expr)                                                        \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      ::mlstm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                         __FILE__, __LINE__);                                         \
      return (int)_e;                                                                 \
    }                                                                                 \
  } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------
// element conversion
// ---------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T x);
template <> __device__ __forceinline__ float to_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }
template <> __device__ __forceinline__ float to_f32<__half>(__half x) { return __half2float(x); }

template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }
template <> __device__ __forceinline__ __half from_f32<__half>(float x) { return __float2half_rn(x); }

// two fp32 values <-> one 32-bit word holding two 16-bit elements (element 0 in the low half)
template <typename T>
__device__ __forceinline__ uint32_t pack2(float a, float b);
template <>
__device__ __forceinline__ uint32_t pack2<__nv_bfloat16>(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
template <>
__device__ __forceinline__ uint32_t pack2<__half>(float a, float b) {
  __half2 v = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
template <typename T>
__device__ __forceinline__ float2 unpack2(uint32_t u);
template <>
__device__ __forceinline__ float2 unpack2<__nv_bfloat16>(uint32_t u) {
  return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
}
template <>
__device__ __forceinline__ float2 unpack2<__half>(uint32_t u) {
  return __half22float2(*reinterpret_cast<__half2*>(&u));
}

// logsigmoid(x) = min(x, 0) - log1p(exp(-|x|))   (reference: F.logsigmoid, native/fw.py:261)
__device__ __forceinline__ float logsigmoid_f32(float x) { return fminf(x, 0.f) - log1pf(expf(-fabsf(x))); }
// sigmoid(-x)  (native/bw.py:323)
__device__ __forceinline__ float sigmoid_neg_f32(float x) { return 1.f / (1.f + expf(x)); }

// ---------------------------------------------------------------------------------------------
// warp-level scans (north_star item 1: forget-gate cumsum and max-state stabilisation)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_incl_sum(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}
__device__ __forceinline__ float warp_incl_max(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v = fmaxf(v, t);
  }
  return v;
}
__device__ __forceinline__ float warp_all_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_all_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Gate vectors of one chunk, computed by ONE warp (all 32 lanes must call).
//   sb[t]  = inclusive cumsum_{r<=t} logsigmoid(f_r)            (vecB,  native/fw.py:261-262)
//   si[t]  = i_t
//   spm[t] = max_{s<=t} (i_s - b_s)   so that   m_t = b_t + max(m_prev, spm[t])  (fw.py:171-184)
// returns g = b_{L-1} (fw.py:82); *amax_rel = max_t (i_t - b_t), i.e. max_t a_t = g + *amax_rel (fw.py:81,83).
// Tokens t >= n_valid (ragged tail) behave like i = -inf, logsigmoid(f) = 0.
constexpr int kMaxChunk = 128;
template <typename T>
__device__ __forceinline__ float chunk_gate_scan(const T* __restrict__ ig, int64_t istride, const T* __restrict__ fg,
                                                 int64_t fstride, int L, int n_valid, float* sb, float* si,
                                                 float* spm, float* amax_rel, bool siging = false) {
  const int lane = threadIdx.x & 31;
  const int E = (L + 31) >> 5;  // consecutive tokens per lane (<= 4)
  float lf[kMaxChunk / 32], iv[kMaxChunk / 32];
  float run = 0.f;
#pragma unroll
  for (int e = 0; e < kMaxChunk / 32; ++e) {
    lf[e] = 0.f;
    iv[e] = -INFINITY;
    if (e < E) {
      int t = lane * E + e;
      if (t < L && t < n_valid) {
        lf[e] = logsigmoid_f32(to_f32<T>(fg[(int64_t)t * fstride]));
        iv[e] = to_f32<T>(ig[(int64_t)t * istride]);
        if (siging) iv[e] = logsigmoid_f32(iv[e]);  // sigmoid input gate (chunkwise_gates.py:34)
      }
      run += lf[e];
      lf[e] = run;  // lane-local inclusive prefix
    }
  }
  float incl = warp_incl_sum(run, lane);
  float base = incl - run;  // exclusive prefix over lanes
  float pmax = -INFINITY;
#pragma unroll
  for (int e = 0; e < kMaxChunk / 32; ++e) {
    if (e < E) {
      lf[e] += base;
      pmax = fmaxf(pmax, iv[e] - lf[e]);
      iv[e] = iv[e];
    }
  }
  // prefix max over lanes of the lane-local maxima
  float incl_max = warp_incl_max(pmax, lane);
  float prev_max = __shfl_up_sync(0xffffffffu, incl_max, 1);
  if (lane == 0) prev_max = -INFINITY;
  float runmax = prev_max;
#pragma unroll
  for (int e = 0; e < kMaxChunk / 32; ++e) {
    if (e < E) {
      int t = lane * E + e;
      runmax = fmaxf(runmax, iv[e] - lf[e]);
      if (t < L) {
        sb[t] = lf[e];
        si[t] = iv[e];
        spm[t] = runmax;
      }
    }
  }
  float g = __shfl_sync(0xffffffffu, incl, 31);
  *amax_rel = warp_all_max(pmax);
  return g;
}

// Dispatch helper: call F<T>() for the runtime dtype.
#define MLSTM_DISPATCH_DTYPE(dtype, T, ...)                       \
  switch (dtype) {                                                \
    case MLSTM_B200_F32: { using T = float; __VA_ARGS__; } break; \
    case MLSTM_B200_BF16: { using T = __nv_bfloat16; __VA_ARGS__; } break; \
    case MLSTM_B200_F16: { using T = __half; __VA_ARGS__; } break; \
    default: ::mlstm::set_error("unknown dtype %d", (int)(dtype)); return MLSTM_B200_EINVAL; \
  }

// launchers implemented in exact_kernels.cu / tensor_kernels.cu
size_t exact_workspace_bytes(const mlstm_b200_shape& s, int backward);
int exact_fw(const mlstm_b200_fw_args& a, cudaStream_t st);
int exact_bw(const mlstm_b200_bw_args& a, cudaStream_t st);

bool tensor_supported(const mlstm_b200_shape& s, int backward);
size_t tensor_workspace_bytes(const mlstm_b200_shape& s, int backward);
size_t tensor_states_bytes(const mlstm_b200_shape& s);
void tensor_set_clock_buffer(void* dev_ptr);
bool tensor_context_is_current();  // a CUDA context is current on the calling thread (driver-level query)
bool tensor_fw_views_ok(const mlstm_b200_fw_args& a);
bool tensor_bw_views_ok(const mlstm_b200_bw_args& a);
int tensor_fw(const mlstm_b200_fw_args& a, cudaStream_t st);
int tensor_fw_epilogue_clusters(const mlstm_b200_shape& s);
int tensor_bw(const mlstm_b200_bw_args& a, cudaStream_t st);


// recurrent step / sequence (step_kernels.cu)
int recurrent_sequence(const mlstm_b200_recurrent_args& a, cudaStream_t st);

// cell output stage (cell_kernels.cu)
size_t cellout_workspace_bytes(const mlstm_b200_cellout_args& a);
int cellout_fw(const mlstm_b200_cellout_args& a, cudaStream_t st);
int cellout_bw(const mlstm_b200_cellout_bw_args& a, cudaStream_t st);
size_t rmsnorm_workspace_bytes(const mlstm_b200_rmsnorm_args& a);
int rmsnorm_fw(const mlstm_b200_rmsnorm_args& a, cudaStream_t st);
int rmsnorm_bw(const mlstm_b200_rmsnorm_bw_args& a, cudaStream_t st);
int convert16(const void* src, void* dst, int64_t n, int src_dtype, int dst_dtype, cudaStream_t st);

}  // namespace mlstm
