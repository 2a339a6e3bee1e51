// The mLSTM cell's output stage, fused: MultiHeadLayerNorm over every (token, head) group of h, the
// (B,NH,S,D) -> (B,S,NH*D) relayout, and ViLLayer's learnable skip, in one pass over HBM each way.
//
//   y[b,s,c] = (h[b,hd,s,d] - mean) * rstd * weight[c] + bias[c] + skip[c] * x[b,s,c],   c = hd*D + d
//
// Reference (what this replaces, paths relative to the reference root):
//   MultiHeadLayerNorm.forward        ultralytics/nn/modules/vision_lstm/vision_lstm2.py:928-944
//       (transpose -> reshape copy -> F.group_norm(num_groups=NH) -> view -> transpose)
//   MatrixLSTMCell.forward tail       vision_lstm2.py:749-751  (h.to(dtype), outnorm, transpose + reshape copy)
//   ViLLayer.mlstm_branch skip add    vision_lstm2.py:306      (h + learnable_skip * x_qk_conv_act)
// and their autograd backward (native_group_norm_backward + the copies), SURVEY.md section 8(f) #3.
//
// HBM-bound elementwise + small-group reduction work: no tensor cores.  One warp covers 128 consecutive
// channels of one token row (4 channels per lane: 8-byte loads for 16-bit types), so x / y / dy / dx move
// as fully coalesced 256-byte warp transactions and every h / dh access is one whole head row.  A row whose
// width H is not a multiple of 128 ends in a tail warp covering H mod 128 (= 32, 64 or 96) channels: its lanes
// past the row's end load and store nothing (TAIL instantiations; D divides 128, so no head straddles two
// warps and the idle lanes form whole head groups of their own).  Group
// statistics are xor-shuffle reductions over the D/4 lanes of a head; the per-channel parameter gradients
// stay in registers across a persistent row loop and are reduced deterministically in two stages
// (CTA partials in the caller's workspace, then one small kernel) -- no atomics.
#include "common.cuh"

namespace mlstm {
namespace {

#ifndef MLSTM_CELL_FW_ROWS
#define MLSTM_CELL_FW_ROWS 4
#endif
#ifndef MLSTM_CELL_BW_ROWS
#define MLSTM_CELL_BW_ROWS 3
#endif
constexpr int kFwRows = MLSTM_CELL_FW_ROWS, kBwRows = MLSTM_CELL_BW_ROWS;  // (fewer for 32-bit operands)  // rows per warp per pipeline stage (two stages are in registers)
constexpr int kMaxWarps = 16;

struct CellP {
  int B, NH, S, D, H, W, lpg;  // H = NH*D channels, W = ceil(H/128) warps per token row, lpg = D/4 lanes per head
  float eps, inv_d;
  const void *h, *x, *dy;
  void *y, *dh, *dx;
  int64_t hs[3], xs[2], ys[2], dys[2], dhs[3], dxs[2];
  const float *weight, *bias, *skip;
  float* partial;  // [gridDim.x][3][H]
};

// Four consecutive elements as they sit in memory; converted to fp32 only where they are consumed, so that the
// software pipeline below really leaves the loads in flight (a conversion placed at the load would wait for it).
template <typename T> struct Raw4 { using type = uint2; };
template <> struct Raw4<float> { using type = float4; };
template <typename T> __device__ __forceinline__ typename Raw4<T>::type ldraw(const T* p) {
  return __ldg(reinterpret_cast<const typename Raw4<T>::type*>(p));
}
template <typename T> __device__ __forceinline__ typename Raw4<T>::type zraw();
template <> __device__ __forceinline__ uint2 zraw<__nv_bfloat16>() { return make_uint2(0u, 0u); }
template <> __device__ __forceinline__ uint2 zraw<__half>() { return make_uint2(0u, 0u); }
template <> __device__ __forceinline__ float4 zraw<float>() { return make_float4(0.f, 0.f, 0.f, 0.f); }
template <typename T> __device__ __forceinline__ void cvt4(const typename Raw4<T>::type& v, float (&o)[4]);
template <> __device__ __forceinline__ void cvt4<float>(const float4& v, float (&o)[4]) {
  o[0] = v.x, o[1] = v.y, o[2] = v.z, o[3] = v.w;
}
template <> __device__ __forceinline__ void cvt4<__nv_bfloat16>(const uint2& v, float (&o)[4]) {
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.y));
  o[0] = a.x, o[1] = a.y, o[2] = b.x, o[3] = b.y;
}
template <> __device__ __forceinline__ void cvt4<__half>(const uint2& v, float (&o)[4]) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
  o[0] = a.x, o[1] = a.y, o[2] = b.x, o[3] = b.y;
}
template <typename T> __device__ __forceinline__ void store4(T* p, const float (&o)[4]);
template <> __device__ __forceinline__ void store4<float>(float* p, const float (&o)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(o[0], o[1], o[2], o[3]);
}
template <> __device__ __forceinline__ void store4<__nv_bfloat16>(__nv_bfloat16* p, const float (&o)[4]) {
  uint2 v;
  *reinterpret_cast<__nv_bfloat162*>(&v.x) = __floats2bfloat162_rn(o[0], o[1]);
  *reinterpret_cast<__nv_bfloat162*>(&v.y) = __floats2bfloat162_rn(o[2], o[3]);
  *reinterpret_cast<uint2*>(p) = v;
}
template <> __device__ __forceinline__ void store4<__half>(__half* p, const float (&o)[4]) {
  uint2 v;
  *reinterpret_cast<__half2*>(&v.x) = __floats2half2_rn(o[0], o[1]);
  *reinterpret_cast<__half2*>(&v.y) = __floats2half2_rn(o[2], o[3]);
  *reinterpret_cast<uint2*>(p) = v;
}

// sum over the LPG lanes that share a head (LPG = D/4 in {8, 16, 32}; groups are lane-aligned)
template <int LPG> __device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = LPG >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// mean / rstd of one head row held 4 elements per lane (two-pass in registers, biased variance as
// F.group_norm: vision_lstm2.py:935-941)
template <int LPG>
__device__ __forceinline__ void group_stats(const float (&hv)[4], float inv_d, float eps, float& mean, float& rstd) {
  mean = group_sum<LPG>(hv[0] + hv[1] + hv[2] + hv[3]) * inv_d;
  float q = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) q += (hv[e] - mean) * (hv[e] - mean);
  rstd = rsqrtf(group_sum<LPG>(q) * inv_d + eps);
}

// Walks the token rows row0, row0 + step, ... of one warp, keeping (batch, position) without a division per row.
// Also carries the running element offsets of the row in the (B, NH, S, D)-strided tensors ("a": stride sb_a per
// batch, ss_a per token) and in the (B, S, H)-strided ones ("c"), advanced by additions only.
struct RowIt {
  int64_t row, rows, step, off_a, off_c, step_a, step_c, wrap_a, wrap_c;
  int si, S, step_s;
  __device__ __forceinline__ RowIt(int64_t row0, int64_t rows_, int64_t step_, int S_, int64_t sb_a, int64_t ss_a,
                                   int64_t sb_c, int64_t ss_c)
      : row(row0), rows(rows_), step(step_), S(S_) {
    const int64_t bi = row0 / S_, step_b = step_ / S_;
    si = (int)(row0 - bi * S_), step_s = (int)(step_ - step_b * S_);
    off_a = bi * sb_a + si * ss_a, off_c = bi * sb_c + si * ss_c;
    step_a = step_b * sb_a + step_s * ss_a, step_c = step_b * sb_c + step_s * ss_c;
    wrap_a = sb_a - S_ * ss_a, wrap_c = sb_c - S_ * ss_c;  // si -= S, ++bi
  }
  __device__ __forceinline__ bool valid() const { return row < rows; }
  __device__ __forceinline__ void next() {
    row += step, si += step_s, off_a += step_a, off_c += step_c;
    if (si >= S) si -= S, off_a += wrap_a, off_c += wrap_c;
  }
};

template <typename TH, typename TX, int U> struct FwRegs {
  typename Raw4<TH>::type hv[U];
  typename Raw4<TX>::type xv[U];
  int64_t yoff[U];  // < 0: no row
};

// Software-pipelined persistent loop: the loads of the next U rows are in flight while the current U rows are
// normalised and stored (two register sets, ping-pong), so every warp keeps U*(h + x) loads outstanding.
template <typename TH, typename TX, int U, int LPG, bool TAIL = false>
__global__ void __launch_bounds__(kMaxWarps * 32, 1) k_cellout_fw(const CellP p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = warp % p.W, r = warp / p.W, R = (blockDim.x >> 5) / p.W;
  const int c0 = slot * 128 + lane * 4, head = c0 / p.D, d0 = c0 % p.D;
  const bool act = !TAIL || c0 < p.H;  // lane inside the row (idle lanes still walk the rows: the shuffles need them)
  float w[4], b[4], sk[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    w[e] = act && p.weight ? p.weight[c0 + e] : 1.f;
    b[e] = act && p.bias ? p.bias[c0 + e] : 0.f;
    sk[e] = act && p.skip ? p.skip[c0 + e] : 0.f;
  }
  const TH* hp = reinterpret_cast<const TH*>(p.h) + head * p.hs[1] + d0;
  const TX* xp = reinterpret_cast<const TX*>(p.x);
  TX* yp = reinterpret_cast<TX*>(p.y);
  RowIt it((int64_t)blockIdx.x * R + r, (int64_t)p.B * p.S, (int64_t)gridDim.x * R, p.S, p.hs[0], p.hs[2], p.ys[0], p.ys[1]);

  using Regs = FwRegs<TH, TX, U>;
  auto load = [&](Regs& g) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      g.yoff[u] = -1;
      g.hv[u] = zraw<TH>(), g.xv[u] = zraw<TX>();
      if (it.valid()) {
        if (act) {
          g.hv[u] = ldraw<TH>(hp + it.off_a);
          if (xp) g.xv[u] = ldraw<TX>(xp + it.off_c + c0);  // x shares y's strides (checked on the host)
        }
        g.yoff[u] = it.off_c + c0;
      }
      it.next();
    }
  };
  auto process = [&](const Regs& g) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float mean, rstd, o[4], hv[4], xv[4];
      cvt4<TH>(g.hv[u], hv);
      cvt4<TX>(g.xv[u], xv);
      group_stats<LPG>(hv, p.inv_d, p.eps, mean, rstd);  // row validity is warp-uniform
#pragma unroll
      for (int e = 0; e < 4; ++e) o[e] = (hv[e] - mean) * rstd * w[e] + b[e] + sk[e] * xv[e];
      if (act && g.yoff[u] >= 0) store4<TX>(yp + g.yoff[u], o);
    }
  };
  Regs ga, gb;
  load(ga);
  while (ga.yoff[0] >= 0) {
    load(gb);
    process(ga);
    if (gb.yoff[0] < 0) break;
    load(ga);
    process(gb);
  }
}

template <typename TH, typename TX, int U> struct BwRegs {
  typename Raw4<TH>::type hv[U];
  typename Raw4<TX>::type xv[U], gv[U];
  int64_t oa[U], oc[U];  // element offsets of the row in h / dh and in dy / x / dx; oa < 0: no row
};

template <typename TH, typename TX, int U, int LPG, bool TAIL = false>
__global__ void __launch_bounds__(kMaxWarps * 32, 1) k_cellout_bw(const CellP p) {
  __shared__ float red[3][kMaxWarps][128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = warp % p.W, r = warp / p.W, R = (blockDim.x >> 5) / p.W;
  const int c0 = slot * 128 + lane * 4, head = c0 / p.D, d0 = c0 % p.D;
  const bool act = !TAIL || c0 < p.H;  // as in the forward; idle lanes accumulate zeros
  float w[4], sk[4], aw[4] = {0.f, 0.f, 0.f, 0.f}, ab[4] = {0.f, 0.f, 0.f, 0.f}, as[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    w[e] = act && p.weight ? p.weight[c0 + e] : 1.f;
    sk[e] = act && p.skip ? p.skip[c0 + e] : 0.f;
  }
  const TH* hp = reinterpret_cast<const TH*>(p.h) + head * p.hs[1] + d0;
  TH* dhp = reinterpret_cast<TH*>(p.dh) + head * p.hs[1] + d0;
  const TX* xp = reinterpret_cast<const TX*>(p.x);
  const TX* dyp = reinterpret_cast<const TX*>(p.dy);
  TX* dxp = reinterpret_cast<TX*>(p.dx);
  RowIt it((int64_t)blockIdx.x * R + r, (int64_t)p.B * p.S, (int64_t)gridDim.x * R, p.S, p.hs[0], p.hs[2], p.dys[0], p.dys[1]);

  using Regs = BwRegs<TH, TX, U>;
  auto load = [&](Regs& g) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      g.oa[u] = -1, g.oc[u] = 0;
      g.hv[u] = zraw<TH>(), g.xv[u] = zraw<TX>(), g.gv[u] = zraw<TX>();
      if (it.valid()) {
        g.oa[u] = it.off_a, g.oc[u] = it.off_c + c0;  // dh shares h's strides, x / dx share dy's (host-checked)
        if (act) {
          g.hv[u] = ldraw<TH>(hp + it.off_a);
          g.gv[u] = ldraw<TX>(dyp + g.oc[u]);
          if (xp) g.xv[u] = ldraw<TX>(xp + g.oc[u]);
        }
      }
      it.next();
    }
  };
  auto process = [&](const Regs& g) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float mean, rstd, xh[4], gw[4], o[4], hv[4], xv[4], gv[4];
      cvt4<TH>(g.hv[u], hv);
      cvt4<TX>(g.xv[u], xv);
      cvt4<TX>(g.gv[u], gv);
      group_stats<LPG>(hv, p.inv_d, p.eps, mean, rstd);
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        xh[e] = (hv[e] - mean) * rstd;
        gw[e] = gv[e] * w[e];
        s1 += gw[e];
        s2 += gw[e] * xh[e];
        aw[e] += gv[e] * xh[e];  // absent rows hold zeros
        ab[e] += gv[e];
        as[e] += gv[e] * xv[e];
      }
      s1 = group_sum<LPG>(s1) * p.inv_d;
      s2 = group_sum<LPG>(s2) * p.inv_d;
      if (act && g.oa[u] >= 0) {
#pragma unroll
        for (int e = 0; e < 4; ++e) o[e] = rstd * (gw[e] - s1 - xh[e] * s2);
        store4<TH>(dhp + g.oa[u], o);
        if (dxp) {
#pragma unroll
          for (int e = 0; e < 4; ++e) o[e] = gv[e] * sk[e];
          store4<TX>(dxp + g.oc[u], o);
        }
      }
    }
  };
  {
    Regs ga, gb;
    load(ga);
    while (ga.oa[0] >= 0) {
      load(gb);
      process(ga);
      if (gb.oa[0] < 0) break;
      load(ga);
      process(gb);
    }
  }
  // stage 1 of the parameter-gradient reduction: over the R row-warps of this CTA
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    red[0][warp][lane * 4 + e] = aw[e];
    red[1][warp][lane * 4 + e] = ab[e];
    red[2][warp][lane * 4 + e] = as[e];
  }
  __syncthreads();
  if (r == 0 && act) {
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int rr = 0; rr < R; ++rr) {
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[e] += red[q][rr * p.W + slot][lane * 4 + e];
      }
      store4<float>(p.partial + ((int64_t)blockIdx.x * 3 + q) * p.H + c0, acc);
    }
  }
}

// stage 2: over CTAs, in a fixed order: one warp per output element, lane l sums partials l, l + 32, ... and the
// lanes are combined by a shuffle tree (same association every run: bit-identical results)
__global__ void k_cellout_reduce(const float* __restrict__ partial, int n_cta, int H, float* dweight, float* dbias, float* dskip) {
  const int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (idx >= 3 * H) return;  // warp-uniform
  const int q = idx / H, c = idx - q * H;
  float* out = q == 0 ? dweight : q == 1 ? dbias : dskip;
  if (!out) return;
  float acc = 0.f;
  for (int i = lane; i < n_cta; i += 32) acc += partial[((int64_t)i * 3 + q) * H + c];
  acc = warp_all_sum(acc);
  if (lane == 0) out[c] = acc;
}

// ---------------------------------------------------------------------------------------------
// RMSNorm in front of the branch (ViLLayer.norm / .ffn_norm = nn.RMSNorm(dim, eps=1e-6), vision_lstm2.py:277-278,
// applied at :318-327).  Under fp16 autocast the input is 16-bit and the weight fp32, so torch.rms_norm falls off
// its fused path ("Mismatch dtype between input and weight") onto a composite of ~15 elementwise / reduction
// kernels per call, forward + backward -- 60 calls per step.  One warp per token row, J = dim/64 element pairs
// per lane (coalesced 128-byte warp accesses), fp32 statistics and arithmetic with ONE rounding at the store, which
// is what the composite does (y = cast((x * rstd) * weight)); the backward keeps the per-channel weight gradient
// in registers and reduces it in two deterministic stages like the cell output stage.
template <typename T> __device__ __forceinline__ float2 ld_pair(const T* p);
template <> __device__ __forceinline__ float2 ld_pair<float>(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }
template <> __device__ __forceinline__ float2 ld_pair<__half>(const __half* p) {
  const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(p));
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
template <> __device__ __forceinline__ float2 ld_pair<__nv_bfloat16>(const __nv_bfloat16* p) {
  const uint32_t u = __ldg(reinterpret_cast<const uint32_t*>(p));
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
}
template <typename T> __device__ __forceinline__ void st_pair(T* p, float a, float b);
template <> __device__ __forceinline__ void st_pair<float>(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
template <> __device__ __forceinline__ void st_pair<__half>(__half* p, float a, float b) { *reinterpret_cast<__half2*>(p) = __floats2half2_rn(a, b); }
template <> __device__ __forceinline__ void st_pair<__nv_bfloat16>(__nv_bfloat16* p, float a, float b) {
  *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b);
}

struct RmsP {
  int64_t rows;
  int C;
  float eps;
  const void *x, *dy;
  void *y, *dx;
  const float* w;
  float* rstd;     // (rows) saved by the forward
  float* partial;  // [gridDim.x][C]
};

template <typename TX, typename TY, int J>
__global__ void __launch_bounds__(512, 1) k_rmsnorm_fw(const RmsP p) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nwarp = (int64_t)gridDim.x * (blockDim.x >> 5);
  float2 w[J];
#pragma unroll
  for (int j = 0; j < J; ++j) w[j] = p.w ? *reinterpret_cast<const float2*>(p.w + 2 * (lane + 32 * j)) : make_float2(1.f, 1.f);
  const float inv_c = 1.f / (float)p.C;
  for (int64_t r0 = warp; r0 < p.rows; r0 += 2 * nwarp) {  // two rows per iteration: their loads overlap
    float2 xa[J], xb[J];
    const int64_t r1 = r0 + nwarp;
    const bool has_b = r1 < p.rows;
    const TX* pa = reinterpret_cast<const TX*>(p.x) + r0 * p.C;
    const TX* pb = reinterpret_cast<const TX*>(p.x) + (has_b ? r1 : r0) * p.C;
#pragma unroll
    for (int j = 0; j < J; ++j) xa[j] = ld_pair<TX>(pa + 2 * (lane + 32 * j));
#pragma unroll
    for (int j = 0; j < J; ++j) xb[j] = ld_pair<TX>(pb + 2 * (lane + 32 * j));
    float sa = 0.f, sb = 0.f;
#pragma unroll
    for (int j = 0; j < J; ++j) sa += xa[j].x * xa[j].x + xa[j].y * xa[j].y, sb += xb[j].x * xb[j].x + xb[j].y * xb[j].y;
    sa = warp_all_sum(sa), sb = warp_all_sum(sb);
    const float ra = rsqrtf(sa * inv_c + p.eps), rb = rsqrtf(sb * inv_c + p.eps);
    TY* ya = reinterpret_cast<TY*>(p.y) + r0 * p.C;
    TY* yb = reinterpret_cast<TY*>(p.y) + r1 * p.C;
#pragma unroll
    for (int j = 0; j < J; ++j)
      st_pair<TY>(ya + 2 * (lane + 32 * j), xa[j].x * ra * w[j].x, xa[j].y * ra * w[j].y);
    if (has_b) {
#pragma unroll
      for (int j = 0; j < J; ++j)
        st_pair<TY>(yb + 2 * (lane + 32 * j), xb[j].x * rb * w[j].x, xb[j].y * rb * w[j].y);
    }
    if (lane == 0) {
      p.rstd[r0] = ra;
      if (has_b) p.rstd[r1] = rb;
    }
  }
}

template <typename TX, typename TY, int J>
__global__ void __launch_bounds__(512, 1) k_rmsnorm_bw(const RmsP p) {
  extern __shared__ float red[];  // [warps][C]
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int64_t warp = (int64_t)blockIdx.x * nw + wib, nwarp = (int64_t)gridDim.x * nw;
  float2 w[J], acc[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    w[j] = p.w ? *reinterpret_cast<const float2*>(p.w + 2 * (lane + 32 * j)) : make_float2(1.f, 1.f);
    acc[j] = make_float2(0.f, 0.f);
  }
  const float inv_c = 1.f / (float)p.C;
  for (int64_t r = warp; r < p.rows; r += nwarp) {
    const TX* px = reinterpret_cast<const TX*>(p.x) + r * p.C;
    const TY* pg = reinterpret_cast<const TY*>(p.dy) + r * p.C;
    float2 x[J], g[J];
#pragma unroll
    for (int j = 0; j < J; ++j) x[j] = ld_pair<TX>(px + 2 * (lane + 32 * j));
#pragma unroll
    for (int j = 0; j < J; ++j) g[j] = ld_pair<TY>(pg + 2 * (lane + 32 * j));
    const float rs = p.rstd[r];
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const float hx = x[j].x * rs, hy = x[j].y * rs;
      acc[j].x += g[j].x * hx;  // d/dw of (x rstd) * w
      acc[j].y += g[j].y * hy;
      g[j].x *= w[j].x, g[j].y *= w[j].y;     // gradient w.r.t. the normalised row
      dot += g[j].x * hx + g[j].y * hy;
      x[j].x = hx, x[j].y = hy;
    }
    dot = warp_all_sum(dot) * inv_c;
    TX* pd = reinterpret_cast<TX*>(p.dx) + r * p.C;
#pragma unroll
    for (int j = 0; j < J; ++j) st_pair<TX>(pd + 2 * (lane + 32 * j), rs * (g[j].x - x[j].x * dot), rs * (g[j].y - x[j].y * dot));
  }
#pragma unroll
  for (int j = 0; j < J; ++j) *reinterpret_cast<float2*>(red + wib * p.C + 2 * (lane + 32 * j)) = acc[j];
  __syncthreads();
  for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
    float a = 0.f;
    for (int k = 0; k < nw; ++k) a += red[k * p.C + c];
    p.partial[(int64_t)blockIdx.x * p.C + c] = a;
  }
}

// Every other width (C a multiple of 32, 64 <= C <= 2048): the row as m = C/32 slots of 32 consecutive channels, one
// element per lane and slot (64-byte warp accesses for 16-bit types, 128-byte for fp32).  A team of T warps shares a
// row, warp t taking slots t, t + T, t + 2T, ... (at most K of them), so no lane holds more than K elements of a row
// whatever C is: registers stay bounded at C = 2048 (K = 16, T = 4).  The team combines its warps' sums through
// shared memory and one named barrier per row (double-buffered by row parity, so one barrier is enough: a warp
// rewrites a buffer only after the whole team has passed the next barrier, i.e. has read it).  The arithmetic is
// the pair kernels': fp32 statistics, one rounding at the store.  T = 1 needs no barrier at all.
template <int T>
__device__ __forceinline__ float team_sum(float v, float* tsum, int wib, int tib) {  // v: this warp's sum (warp-uniform)
  if constexpr (T == 1) {
    return v;
  } else {
    if ((threadIdx.x & 31) == 0) tsum[wib] = v;
    asm volatile("bar.sync %0, %1;" ::"r"(1 + tib), "r"(T * 32) : "memory");
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < T; ++i) s += tsum[tib * T + i];  // same order in every warp of the team
    return s;
  }
}

template <typename TX, typename TY, int K, int T>
__global__ void __launch_bounds__(512, 1) k_rmsnorm_fw_slots(const RmsP p) {
  __shared__ float tsum[2][2][16];  // [row parity][row a / b][warp]
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, t = wib % T, tib = wib / T;
  const int teams = (blockDim.x >> 5) / T, m = p.C >> 5;
  const int64_t team = (int64_t)blockIdx.x * teams + tib, nteam = (int64_t)gridDim.x * teams;
  float w[K];
#pragma unroll
  for (int k = 0; k < K; ++k) w[k] = (k * T + t < m && p.w) ? p.w[(k * T + t) * 32 + lane] : 1.f;
  const float inv_c = 1.f / (float)p.C;
  const int64_t c0 = t * 32 + lane;
  int par = 0;
  for (int64_t r0 = team; r0 < p.rows; r0 += 2 * nteam, par ^= 1) {  // two rows per iteration: their loads overlap
    float xa[K], xb[K];
    const int64_t r1 = r0 + nteam;
    const bool has_b = r1 < p.rows;
    const TX* pa = reinterpret_cast<const TX*>(p.x) + r0 * p.C + c0;
    const TX* pb = reinterpret_cast<const TX*>(p.x) + (has_b ? r1 : r0) * p.C + c0;
#pragma unroll
    for (int k = 0; k < K; ++k) xa[k] = k * T + t < m ? to_f32<TX>(__ldg(pa + k * T * 32)) : 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) xb[k] = k * T + t < m ? to_f32<TX>(__ldg(pb + k * T * 32)) : 0.f;
    float sa = 0.f, sb = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) sa += xa[k] * xa[k], sb += xb[k] * xb[k];
    sa = team_sum<T>(warp_all_sum(sa), tsum[par][0], wib, tib);
    sb = team_sum<T>(warp_all_sum(sb), tsum[par][1], wib, tib);
    const float ra = rsqrtf(sa * inv_c + p.eps), rb = rsqrtf(sb * inv_c + p.eps);
    TY* ya = reinterpret_cast<TY*>(p.y) + r0 * p.C + c0;
    TY* yb = reinterpret_cast<TY*>(p.y) + r1 * p.C + c0;
#pragma unroll
    for (int k = 0; k < K; ++k)
      if (k * T + t < m) ya[k * T * 32] = from_f32<TY>(xa[k] * ra * w[k]);
    if (has_b) {
#pragma unroll
      for (int k = 0; k < K; ++k)
        if (k * T + t < m) yb[k * T * 32] = from_f32<TY>(xb[k] * rb * w[k]);
    }
    if (t == 0 && lane == 0) {
      p.rstd[r0] = ra;
      if (has_b) p.rstd[r1] = rb;
    }
  }
}

// Dynamic shared memory: (16 / T) teams x C floats <= 32 KB for every C (T = ceil(C / 512) rounded up to 1, 2, 4).
template <typename TX, typename TY, int K, int T>
__global__ void __launch_bounds__(512, 1) k_rmsnorm_bw_slots(const RmsP p) {
  extern __shared__ float red[];    // [teams][C]
  __shared__ float tsum[2][16];     // [row parity][warp]
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, t = wib % T, tib = wib / T;
  const int teams = (blockDim.x >> 5) / T, m = p.C >> 5;
  const int64_t team = (int64_t)blockIdx.x * teams + tib, nteam = (int64_t)gridDim.x * teams;
  float w[K], acc[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    w[k] = (k * T + t < m && p.w) ? p.w[(k * T + t) * 32 + lane] : 1.f;
    acc[k] = 0.f;
  }
  const float inv_c = 1.f / (float)p.C;
  const int64_t c0 = t * 32 + lane;
  int par = 0;
  for (int64_t r = team; r < p.rows; r += nteam, par ^= 1) {
    const TX* px = reinterpret_cast<const TX*>(p.x) + r * p.C + c0;
    const TY* pg = reinterpret_cast<const TY*>(p.dy) + r * p.C + c0;
    float x[K], g[K];
#pragma unroll
    for (int k = 0; k < K; ++k) x[k] = k * T + t < m ? to_f32<TX>(__ldg(px + k * T * 32)) : 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) g[k] = k * T + t < m ? to_f32<TY>(__ldg(pg + k * T * 32)) : 0.f;
    const float rs = p.rstd[r];
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float hx = x[k] * rs;
      acc[k] += g[k] * hx;  // d/dw of (x rstd) * w
      g[k] *= w[k];         // gradient w.r.t. the normalised row
      dot += g[k] * hx;
      x[k] = hx;
    }
    dot = team_sum<T>(warp_all_sum(dot), tsum[par], wib, tib) * inv_c;
    TX* pd = reinterpret_cast<TX*>(p.dx) + r * p.C + c0;
#pragma unroll
    for (int k = 0; k < K; ++k)
      if (k * T + t < m) pd[k * T * 32] = from_f32<TX>(rs * (g[k] - x[k] * dot));
  }
#pragma unroll
  for (int k = 0; k < K; ++k)
    if (k * T + t < m) red[tib * p.C + (k * T + t) * 32 + lane] = acc[k];
  __syncthreads();
  for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
    float a = 0.f;
    for (int q = 0; q < teams; ++q) a += red[q * p.C + c];
    p.partial[(int64_t)blockIdx.x * p.C + c] = a;
  }
}

__global__ void k_rmsnorm_reduce(const float* __restrict__ partial, int n_cta, int C, float* dw) {
  const int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (idx >= C) return;
  float acc = 0.f;
  for (int i = lane; i < n_cta; i += 32) acc += partial[(int64_t)i * C + idx];
  acc = warp_all_sum(acc);
  if (lane == 0) dw[idx] = acc;
}

int grid_ctas() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return 2 * sms;  // two short CTAs per SM's worth of rows: evens out the tail without extra partials
}

bool aligned(const void* p, size_t a) { return ((uintptr_t)p % a) == 0; }

int fill(const mlstm_b200_cellout_args& a, CellP& p) {
  if (a.B <= 0 || a.NH <= 0 || a.S <= 0 || a.D <= 0) {
    set_error("cellout: bad shape B=%d NH=%d S=%d D=%d", a.B, a.NH, a.S, a.D);
    return MLSTM_B200_EINVAL;
  }
  const int H = a.NH * a.D;
  if ((a.D != 32 && a.D != 64 && a.D != 128) || H > kMaxWarps * 128) {
    set_error("cellout: needs D in {32,64,128} and NH*D <= %d (got D=%d NH=%d)", kMaxWarps * 128, a.D, a.NH);
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (!a.h.ptr || a.h.stride[3] != 1) {
    set_error("cellout: h is NULL or its innermost stride is not 1");
    return MLSTM_B200_EINVAL;
  }
  if (a.x.ptr && (!a.skip || a.x.stride[2] != 1)) {
    set_error("cellout: x needs a skip vector and a unit innermost stride");
    return MLSTM_B200_EINVAL;
  }
  p.B = a.B, p.NH = a.NH, p.S = a.S, p.D = a.D, p.H = H, p.W = (H + 127) / 128, p.lpg = a.D / 4;
  p.eps = a.eps, p.inv_d = 1.f / (float)a.D;
  p.h = a.h.ptr, p.x = a.x.ptr;
  for (int i = 0; i < 3; ++i) p.hs[i] = a.h.stride[i];
  for (int i = 0; i < 2; ++i) p.xs[i] = a.x.stride[i];
  p.weight = a.weight, p.bias = a.bias, p.skip = a.x.ptr ? a.skip : nullptr;
  return 0;
}

bool vec_ok(const mlstm_b200_tensor& t, int nstride, int dtype) {
  const size_t bytes = dtype == MLSTM_B200_F32 ? 16 : 8;
  if (!aligned(t.ptr, bytes)) return false;
  for (int i = 0; i < nstride; ++i)
    if (t.stride[i] % 4) return false;
  return true;
}

template <typename F> int dispatch2(int th, int tx, F&& f) {
  // (h dtype, x/y dtype) pairs; 16-bit h is what the mLSTM kernels emit, fp32 h is the exact family's
#define MLSTM_CELL_CASE(A, TA, Bv, TB) \
  if (th == A && tx == Bv) return f(TA{}, TB{});
  MLSTM_CELL_CASE(MLSTM_B200_BF16, __nv_bfloat16, MLSTM_B200_F16, __half)
  MLSTM_CELL_CASE(MLSTM_B200_BF16, __nv_bfloat16, MLSTM_B200_BF16, __nv_bfloat16)
  MLSTM_CELL_CASE(MLSTM_B200_BF16, __nv_bfloat16, MLSTM_B200_F32, float)
  MLSTM_CELL_CASE(MLSTM_B200_F16, __half, MLSTM_B200_F16, __half)
  MLSTM_CELL_CASE(MLSTM_B200_F16, __half, MLSTM_B200_BF16, __nv_bfloat16)
  MLSTM_CELL_CASE(MLSTM_B200_F16, __half, MLSTM_B200_F32, float)
  MLSTM_CELL_CASE(MLSTM_B200_F32, float, MLSTM_B200_F16, __half)
  MLSTM_CELL_CASE(MLSTM_B200_F32, float, MLSTM_B200_BF16, __nv_bfloat16)
  MLSTM_CELL_CASE(MLSTM_B200_F32, float, MLSTM_B200_F32, float)
#undef MLSTM_CELL_CASE
  set_error("cellout: unknown dtype pair (%d, %d)", th, tx);
  return MLSTM_B200_EINVAL;
}

int block_threads(const CellP& p) { return (kMaxWarps / p.W) * p.W * 32; }

}  // namespace

size_t cellout_workspace_bytes(const mlstm_b200_cellout_args& a) {
  return (size_t)grid_ctas() * 3 * (size_t)a.NH * a.D * sizeof(float);
}

int cellout_fw(const mlstm_b200_cellout_args& a, cudaStream_t st) {
  CellP p{};
  if (int e = fill(a, p)) return e;
  if (!a.y.ptr || a.y.stride[2] != 1) {
    set_error("cellout: y is NULL or its innermost stride is not 1");
    return MLSTM_B200_EINVAL;
  }
  if (a.x.ptr && a.x_dtype != a.y_dtype) {
    set_error("cellout: x and y must have the same dtype");
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (!vec_ok(a.h, 3, a.h_dtype) || !vec_ok(a.y, 2, a.y_dtype) || (a.x.ptr && !vec_ok(a.x, 2, a.x_dtype))) {
    set_error("cellout: tensors must be 8-byte (16-bit) / 16-byte (fp32) aligned with strides that are multiples of 4");
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (a.x.ptr && (a.x.stride[0] != a.y.stride[0] || a.x.stride[1] != a.y.stride[1])) {
    set_error("cellout: x and y must have the same strides");
    return MLSTM_B200_EUNSUPPORTED;
  }
  p.y = a.y.ptr;
  for (int i = 0; i < 2; ++i) p.ys[i] = a.y.stride[i];
  const int grid = grid_ctas(), block = block_threads(p);
  int rc = dispatch2(a.h_dtype, a.y_dtype, [&](auto th, auto tx) {
    constexpr int kRows = (sizeof(th) + sizeof(tx)) <= 4 ? kFwRows : kFwRows / 2;
    using TH = decltype(th);
    using TX = decltype(tx);
    switch (p.lpg) {  // (D = 128 rows are always whole warps)
      case 8:
        if (p.H % 128) k_cellout_fw<TH, TX, kRows, 8, true><<<grid, block, 0, st>>>(p);
        else k_cellout_fw<TH, TX, kRows, 8><<<grid, block, 0, st>>>(p);
        break;
      case 16:
        if (p.H % 128) k_cellout_fw<TH, TX, kRows, 16, true><<<grid, block, 0, st>>>(p);
        else k_cellout_fw<TH, TX, kRows, 16><<<grid, block, 0, st>>>(p);
        break;
      default: k_cellout_fw<TH, TX, kRows, 32><<<grid, block, 0, st>>>(p); break;
    }
    return 0;
  });
  if (rc) return rc;
  count_launch(1);
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int cellout_bw(const mlstm_b200_cellout_bw_args& b, cudaStream_t st) {
  const mlstm_b200_cellout_args& a = b.fw;
  CellP p{};
  if (int e = fill(a, p)) return e;
  if (!b.dy.ptr || b.dy.stride[2] != 1 || !b.dh.ptr || b.dh.stride[3] != 1 || (b.dx.ptr && b.dx.stride[2] != 1)) {
    set_error("cellout_bw: dy / dh are NULL or an innermost stride is not 1");
    return MLSTM_B200_EINVAL;
  }
  if (a.x.ptr && a.x_dtype != a.y_dtype) {
    set_error("cellout: x and y must have the same dtype");
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (!vec_ok(a.h, 3, a.h_dtype) || !vec_ok(b.dh, 3, a.h_dtype) || !vec_ok(b.dy, 2, a.y_dtype) ||
      (a.x.ptr && !vec_ok(a.x, 2, a.x_dtype)) || (b.dx.ptr && !vec_ok(b.dx, 2, a.y_dtype))) {
    set_error("cellout_bw: tensors must be 8-byte (16-bit) / 16-byte (fp32) aligned with strides that are multiples of 4");
    return MLSTM_B200_EUNSUPPORTED;
  }
  for (int i = 0; i < 3; ++i) {
    if (b.dh.stride[i] != a.h.stride[i]) {
      set_error("cellout_bw: dh must have the strides of h");
      return MLSTM_B200_EUNSUPPORTED;
    }
  }
  for (int i = 0; i < 2; ++i) {
    if ((a.x.ptr && a.x.stride[i] != b.dy.stride[i]) || (b.dx.ptr && b.dx.stride[i] != b.dy.stride[i])) {
      set_error("cellout_bw: x and dx must have the strides of dy");
      return MLSTM_B200_EUNSUPPORTED;
    }
  }
  const size_t need = cellout_workspace_bytes(a);
  if (!b.workspace || b.workspace_bytes < need) {
    set_error("cellout_bw: workspace too small: need %zu bytes, got %zu", need, b.workspace_bytes);
    return MLSTM_B200_EWORKSPACE;
  }
  p.dy = b.dy.ptr, p.dh = b.dh.ptr, p.dx = b.dx.ptr;
  p.partial = reinterpret_cast<float*>(b.workspace);
  for (int i = 0; i < 2; ++i) p.dys[i] = b.dy.stride[i], p.dxs[i] = b.dx.stride[i];
  for (int i = 0; i < 3; ++i) p.dhs[i] = b.dh.stride[i];
  const int grid = grid_ctas(), block = block_threads(p);
  int rc = dispatch2(a.h_dtype, a.y_dtype, [&](auto th, auto tx) {
    constexpr int kRows = (sizeof(th) + 2 * sizeof(tx)) <= 6 ? kBwRows : 2;  // register budget per pipeline stage
    using TH = decltype(th);
    using TX = decltype(tx);
    switch (p.lpg) {
      case 8:
        if (p.H % 128) k_cellout_bw<TH, TX, kRows, 8, true><<<grid, block, 0, st>>>(p);
        else k_cellout_bw<TH, TX, kRows, 8><<<grid, block, 0, st>>>(p);
        break;
      case 16:
        if (p.H % 128) k_cellout_bw<TH, TX, kRows, 16, true><<<grid, block, 0, st>>>(p);
        else k_cellout_bw<TH, TX, kRows, 16><<<grid, block, 0, st>>>(p);
        break;
      default: k_cellout_bw<TH, TX, kRows, 32><<<grid, block, 0, st>>>(p); break;
    }
    return 0;
  });
  if (rc) return rc;
  MLSTM_CUDA_CHECK(cudaGetLastError());
  k_cellout_reduce<<<(3 * p.H * 32 + 255) / 256, 256, 0, st>>>(p.partial, grid, p.H, b.dweight, b.dbias, b.dskip);
  count_launch(2);
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

size_t rmsnorm_workspace_bytes(const mlstm_b200_rmsnorm_args& a) { return (size_t)grid_ctas() * a.C * sizeof(float); }

namespace {
int rms_check(const mlstm_b200_rmsnorm_args& a) {
  if (a.rows <= 0 || !a.x || !a.rstd) {
    set_error("rmsnorm: bad arguments");
    return MLSTM_B200_EINVAL;
  }
  if (a.C % 32 != 0 || a.C < 64 || a.C > 2048) {
    set_error("rmsnorm: dim %d not covered (a multiple of 32 from 64 to 2048)", a.C);
    return MLSTM_B200_EUNSUPPORTED;
  }
  return 0;
}
template <typename TX, typename TY, int J>
void rms_launch(const RmsP& p, bool backward, cudaStream_t st) {
  const int grid = grid_ctas();
  if (backward)
    k_rmsnorm_bw<TX, TY, J><<<grid, 512, 16 * p.C * sizeof(float), st>>>(p);
  else
    k_rmsnorm_fw<TX, TY, J><<<grid, 512, 0, st>>>(p);
}
template <typename TX, typename TY, int K, int T>
void rms_launch_slots(const RmsP& p, bool backward, cudaStream_t st) {
  const int grid = grid_ctas();
  if (backward)
    k_rmsnorm_bw_slots<TX, TY, K, T><<<grid, 512, (16 / T) * p.C * sizeof(float), st>>>(p);
  else
    k_rmsnorm_fw_slots<TX, TY, K, T><<<grid, 512, 0, st>>>(p);
}
template <typename TX, typename TY>
int rms_dispatch_j(const RmsP& p, bool backward, cudaStream_t st) {
  if (p.C % 64 == 0) {
    switch (p.C / 64) {  // the model widths 192 / 256 / 384 / 512: one element pair per lane and 64 channels
      case 3: rms_launch<TX, TY, 3>(p, backward, st); return 0;
      case 4: rms_launch<TX, TY, 4>(p, backward, st); return 0;
      case 6: rms_launch<TX, TY, 6>(p, backward, st); return 0;
      case 8: rms_launch<TX, TY, 8>(p, backward, st); return 0;
    }
  }
  const int m = p.C / 32;  // every other width (rms_check): 32-channel slots, K per warp, T warps per row
  if (m <= 4) rms_launch_slots<TX, TY, 4, 1>(p, backward, st);
  else if (m <= 8) rms_launch_slots<TX, TY, 8, 1>(p, backward, st);
  else if (m <= 16) rms_launch_slots<TX, TY, 16, 1>(p, backward, st);
  else if (m <= 32) rms_launch_slots<TX, TY, 16, 2>(p, backward, st);
  else rms_launch_slots<TX, TY, 16, 4>(p, backward, st);
  return 0;
}
int rms_dispatch(int tx, int ty, const RmsP& p, bool backward, cudaStream_t st) {
  return dispatch2(tx, ty, [&](auto a, auto b) { return rms_dispatch_j<decltype(a), decltype(b)>(p, backward, st); });
}
}  // namespace

// ---------------------------------------------------------------------------------------------
// 16-bit re-rounding pass: fp16 <-> bf16 over a contiguous buffer.  The reference kernels re-round their inputs to
// autocast_kernel_dtype under CUDA autocast (custom_fwd(cast_inputs=bf16), native/fwbw.py:37); under ultralytics' fp16
// AMP that is one pass over q / k / v per cell.  torch's copy_ does it with its generic unrolled elementwise kernel
// (~3 TB/s here); this one is a plain streaming kernel: 16-byte vectors, four in flight per thread, evict-first loads
// and stores, 4 bytes of HBM traffic per element.  Values go through fp32 (exact for both source formats), one RN
// rounding -- bit-identical to Tensor.to().
template <typename TS, typename TD>
__device__ __forceinline__ uint4 convert8(uint4 v) {
  const uint32_t in[4] = {v.x, v.y, v.z, v.w};
  uint32_t out[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 f = unpack2<TS>(in[j]);
    out[j] = pack2<TD>(f.x, f.y);
  }
  return make_uint4(out[0], out[1], out[2], out[3]);
}

template <typename TS, typename TD>
__global__ void __launch_bounds__(256) k_convert16(const TS* __restrict__ src, TD* __restrict__ dst, int64_t n) {
  const int64_t nvec = n >> 3;
  const uint4* s4 = reinterpret_cast<const uint4*>(src);
  uint4* d4 = reinterpret_cast<uint4*>(dst);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < nvec; i += 4 * stride) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = __ldcs(s4 + i + u * stride);
#pragma unroll
    for (int u = 0; u < 4; ++u) __stcs(d4 + i + u * stride, convert8<TS, TD>(v[u]));
  }
  for (; i < nvec; i += stride) __stcs(d4 + i, convert8<TS, TD>(__ldcs(s4 + i)));
  // tail of fewer than 8 elements
  const int64_t t = (nvec << 3) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) dst[t] = from_f32<TD>(to_f32<TS>(src[t]));
}

template <typename TS, typename TD>
__global__ void __launch_bounds__(256) k_convert16_scalar(const TS* __restrict__ src, TD* __restrict__ dst, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = from_f32<TD>(to_f32<TS>(src[i]));
}

template <typename TS, typename TD>
void launch_convert16(const void* src, void* dst, int64_t n, cudaStream_t st) {
  const int64_t per_cta = 256 * 8 * 4;
  const int64_t want = (n + per_cta - 1) / per_cta;
  const int grid = (int)(want < 1 ? 1 : (want > 8 * (grid_ctas() / 2) ? 8 * (grid_ctas() / 2) : want));
  if (aligned(src, 16) && aligned(dst, 16))
    k_convert16<TS, TD><<<grid, 256, 0, st>>>((const TS*)src, (TD*)dst, n);
  else  // views that start inside a vector: element-wise (same values)
    k_convert16_scalar<TS, TD><<<grid, 256, 0, st>>>((const TS*)src, (TD*)dst, n);
}

int convert16(const void* src, void* dst, int64_t n, int src_dtype, int dst_dtype, cudaStream_t st) {
  const bool ok = (src_dtype == MLSTM_B200_F16 && dst_dtype == MLSTM_B200_BF16) ||
                  (src_dtype == MLSTM_B200_BF16 && dst_dtype == MLSTM_B200_F16);
  if (!ok) {
    set_error("convert16: fp16 -> bf16 or bf16 -> fp16 (got dtypes %d -> %d)", src_dtype, dst_dtype);
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (n < 0 || (n > 0 && (!src || !dst))) {
    set_error("convert16: NULL buffer or negative length");
    return MLSTM_B200_EINVAL;
  }
  if (n == 0) return 0;
  if (src_dtype == MLSTM_B200_F16) launch_convert16<__half, __nv_bfloat16>(src, dst, n, st);
  else launch_convert16<__nv_bfloat16, __half>(src, dst, n, st);
  count_launch(1);
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int rmsnorm_fw(const mlstm_b200_rmsnorm_args& a, cudaStream_t st) {
  if (int e = rms_check(a)) return e;
  if (!a.y) {
    set_error("rmsnorm: y is NULL");
    return MLSTM_B200_EINVAL;
  }
  RmsP p{};
  p.rows = a.rows, p.C = a.C, p.eps = a.eps, p.x = a.x, p.y = a.y, p.w = a.weight, p.rstd = a.rstd;
  if (int e = rms_dispatch(a.x_dtype, a.y_dtype, p, false, st)) return e;
  count_launch(1);
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int rmsnorm_bw(const mlstm_b200_rmsnorm_bw_args& b, cudaStream_t st) {
  const mlstm_b200_rmsnorm_args& a = b.fw;
  if (int e = rms_check(a)) return e;
  if (!b.dy || !b.dx) {
    set_error("rmsnorm_bw: dy / dx are NULL");
    return MLSTM_B200_EINVAL;
  }
  const size_t need = rmsnorm_workspace_bytes(a);
  if (!b.workspace || b.workspace_bytes < need) {
    set_error("rmsnorm_bw: workspace too small: need %zu bytes, got %zu", need, b.workspace_bytes);
    return MLSTM_B200_EWORKSPACE;
  }
  RmsP p{};
  p.rows = a.rows, p.C = a.C, p.eps = a.eps, p.x = a.x, p.dy = b.dy, p.dx = b.dx, p.w = a.weight, p.rstd = a.rstd;
  p.partial = reinterpret_cast<float*>(b.workspace);
  if (int e = rms_dispatch(a.x_dtype, a.y_dtype, p, true, st)) return e;
  MLSTM_CUDA_CHECK(cudaGetLastError());
  if (b.dweight) k_rmsnorm_reduce<<<(a.C * 32 + 255) / 256, 256, 0, st>>>(p.partial, grid_ctas(), a.C, b.dweight);
  count_launch(2);
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace mlstm
