// Tensor-core kernel family of the sm_100a mLSTM chunkwise path: tcgen05.mma with TMEM
// accumulators, operands staged by TMA (128B swizzle), one persistent CTA per (batch, head)
// that walks the sequence in 128-token tiles and keeps the C / n / m state on chip
// (C: fp32 master copy in registers + bf16 MMA operand copy in shared memory).
//
// CTA = 8 worker warps + 1 control warp.  Worker warp w owns tile rows 32*(w%4).. (== its TMEM
// lane quadrant) and column half w/4.  The control warp issues every TMA copy and every
// tcgen05.mma (one lane), and runs the gate scans (log-sigmoid cumsum, running max) one tile
// ahead of the workers.  Hand-offs: workers -> control through named barriers (bar.arrive /
// bar.sync), control -> workers through mbarriers (tcgen05.commit, TMA complete_tx).
//
// Forward, per 128-token tile k (math: SURVEY.md Appendix A; reference native/fw.py:29-221):
//   S      = Q K^T                      tcgen05  M128 N128 K64   (A, B K-major from TMA)
//   dC     = (abar.K)^T V               tcgen05  M64  N64  K128  (A, B MN-major)
//   P      = S . scale . exp(b_t - b_s + i_s - m_t), s <= t      (registers, from TMEM)
//   Hintra = P V                        tcgen05  M128 N64  K128  (A = P written swizzled)
//   Hinter = Q C_{k-1}                  tcgen05  M128 N64  K64   (B = bf16 copy of C)
//   h      = (Hintra + bbar.scale.Hinter) / (max(|den|, exp(-m_t)) + eps)   -> TMA store
//   C_k    = gbar C_{k-1} + dC          fp32 registers (the only sequential dependency)
// h and the final states do not depend on the tile length (m_t equals the step-recurrent
// stabiliser), so a 128-token tile is used although the API chunk size is 64.
#include <atomic>
#include <mutex>
#include <set>
#include <type_traits>
#include <utility>

#include "common.cuh"
#include "sm100.cuh"

namespace mlstm {
namespace {

using namespace sm100;

constexpr int LT = 128;           // tokens per tile
constexpr int kWorkers = 256;     // 8 worker warps
constexpr int kTcThreads = 320;   // + control warp (TMA / MMA issue) + scan warp (gate vectors, dF scan)
constexpr int kCtlWarp = 8, kScanWarp = 9;
constexpr int kNbAB = kWorkers + 32;  // workers + control
constexpr int kNbC = kWorkers + 64;   // workers + control + scan
constexpr float kLog2e = 1.4426950408889634f;
enum { NB_A = 1, NB_B = 2, NB_C = 3, NB_PAIR0 = 4 };  // named barriers: operand ready / P ready / epilogue done / warp pairs (4..7)

// per-tile gate vectors produced by the control warp (floats)
struct GateBuf {
  static constexpr int oB = 0, oI = LT, oPm = 2 * LT, oY = 3 * LT, oF = 4 * LT, oMt = 5 * LT, oNt = 6 * LT,
                       oCf = 7 * LT, oDi = 8 * LT, oDf = 9 * LT, oScal = 10 * LT, kFloats = 10 * LT + 8;
  // oScal: 0 g, 1 amax, 2 m_prev, 3 m_next (backward), 4..7 max of y over each 32-column unit
  // oDi / oDf: derivative of the soft cap at the raw gate pre-activations (1 when the cap is off); backward only
};

#ifdef MLSTM_TC_PROFILE  // phase clocks of CTA 0 (tools/phase_clocks.py builds with this flag)
#define TC_PROF(tile, slot) \
  if (p.prof && blockIdx.x == 0 && (threadIdx.x == 0 || threadIdx.x == kWorkers)) p.prof[(tile) * 16 + (slot)] = clock64()
// every CTA's lifetime on the global nanosecond timer: [3300 + 3*cta + {0 entry, 1 exit, 2 SM id}] (cta < 260)
#define TC_PROF_CTA(which)                                                                  \
  if (p.prof && threadIdx.x == 0 && blockIdx.x < 260) {                                    \
    unsigned long long _t;                                                                  \
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_t));                                 \
    p.prof[3300 + 3 * blockIdx.x + (which)] = (long long)_t;                               \
    if ((which) == 0) {                                                                     \
      unsigned _sm;                                                                         \
      asm volatile("mov.u32 %0, %%smid;" : "=r"(_sm));                                     \
      p.prof[3300 + 3 * blockIdx.x + 2] = _sm;                                              \
    }                                                                                       \
  }
#else
#define TC_PROF(tile, slot)
#define TC_PROF_CTA(which)
#endif

// store 32 consecutive columns (col0 multiple of 32) of row `row` of a [128][64]-subtiled,
// 128B-swizzled 16-bit matrix; `base` points at the first subtile, subtiles are LT*128 B apart.
template <typename T>
__device__ __forceinline__ void store_row32(uint8_t* base, int row, int col0, const float (&v)[32]) {
  uint8_t* tile = base + (col0 >> 6) * (LT * 128);
  const int c = col0 & 63;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint4 u;
    u.x = pack2<T>(v[8 * j + 0], v[8 * j + 1]);
    u.y = pack2<T>(v[8 * j + 2], v[8 * j + 3]);
    u.z = pack2<T>(v[8 * j + 4], v[8 * j + 5]);
    u.w = pack2<T>(v[8 * j + 6], v[8 * j + 7]);
    *reinterpret_cast<uint4*>(tile + swz128(row, c + 8 * j)) = u;
  }
}

// Column sums over the 32 rows held by a warp: lane L ends up with sum_rows v[.][L]
// (butterfly transpose-reduce, 31 shuffles).  v is destroyed.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int j = 0; j < off; ++j) {
      const float keep = hi ? v[j + off] : v[j];
      const float send = hi ? v[j] : v[j + off];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

// ---------------------------------------------------------------------------------------------
// Head-dim dependent layout of the [rows][D] 16-bit tiles (Q, K, V, H, C, ...): D = 64 -> 128-byte
// rows, TMA / UMMA SWIZZLE_128B; D = 32 -> 64-byte rows, SWIZZLE_64B (descriptor forms validated by
// tests/cuda/umma_probe.cu sw64).  The 128 x 128 tiles (P, Sb', dS) always use 128-byte rows.
// ---------------------------------------------------------------------------------------------
template <int D>
struct Lay {
  static_assert(D == 64 || D == 32, "head dim 64 or 32");
  static constexpr int kRowB = 2 * D;                  // bytes per tile row
  static constexpr int kTile = LT * kRowB;             // one [128][D] tile
  static constexpr int kState = D * kRowB;             // one [D][D] state tile
  static constexpr uint32_t kSbo = 8 * kRowB;          // 8-row swizzle atom
  static constexpr uint32_t kLt = D == 64 ? 2u : 4u;   // UMMA layout type
  static constexpr int CW = D / 2;                     // columns per worker thread
  static constexpr uint32_t kAdvMN = 16 * kRowB;       // descriptor advance per 16 K-rows of an MN-major operand
  __device__ static __forceinline__ uint32_t swz(int row, int col) { return D == 64 ? swz128(row, col) : swz64(row, col); }
  // K-major operand: lbo = 0; MN-major operand: lbo = byte distance to the next D-wide block (0 re-reads the
  // same block: the M = 64 MMA of the D = 32 state update duplicates its 32 real rows)
  __device__ static __forceinline__ uint64_t desc(uint32_t saddr, uint32_t lbo) { return umma_smem_desc_lt(saddr, lbo, kSbo, kLt); }
};

// store N consecutive columns (col0 multiple of 8) of row `row` of a swizzled [rows][D] 16-bit tile
template <typename T, int D, int N>
__device__ __forceinline__ void store_cols(uint8_t* tile, int row, int col0, const float (&v)[N]) {
#pragma unroll
  for (int j = 0; j < N / 8; ++j) {
    uint4 u;
    u.x = pack2<T>(v[8 * j + 0], v[8 * j + 1]);
    u.y = pack2<T>(v[8 * j + 2], v[8 * j + 3]);
    u.z = pack2<T>(v[8 * j + 4], v[8 * j + 5]);
    u.w = pack2<T>(v[8 * j + 6], v[8 * j + 7]);
    *reinterpret_cast<uint4*>(tile + Lay<D>::swz(row, col0 + 8 * j)) = u;
  }
}

// Column sums over the 32 rows held by a warp for N = 16 columns: every lane ends up with the sum of
// column (lane & 15).
__device__ __forceinline__ float warp_colsum16(float (&v)[16], int lane) {
#pragma unroll
  for (int off = 8; off >= 1; off >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int j = 0; j < off; ++j) {
      const float keep = hi ? v[j + off] : v[j];
      const float send = hi ? v[j] : v[j + off];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}
template <int N>
__device__ __forceinline__ float warp_colsum(float (&v)[N], int lane);
template <>
__device__ __forceinline__ float warp_colsum<32>(float (&v)[32], int lane) { return warp_colsum32(v, lane); }
template <>
__device__ __forceinline__ float warp_colsum<16>(float (&v)[16], int lane) { return warp_colsum16(v, lane); }

// packed 16-bit pair times a 16-bit scalar (one HMUL2)
template <typename T>
__device__ __forceinline__ uint32_t mul2(uint32_t a, T s);
template <>
__device__ __forceinline__ uint32_t mul2<__nv_bfloat16>(uint32_t a, __nv_bfloat16 s) {
  __nv_bfloat162 r = __hmul2(*reinterpret_cast<__nv_bfloat162*>(&a), __bfloat162bfloat162(s));
  return *reinterpret_cast<uint32_t*>(&r);
}
template <>
__device__ __forceinline__ uint32_t mul2<__half>(uint32_t a, __half s) {
  __half2 r = __hmul2(*reinterpret_cast<__half2*>(&a), __half2half2(s));
  return *reinterpret_cast<uint32_t*>(&r);
}
// registers -> TMEM, 16 or 8 consecutive 32-bit columns of this thread's lane
__device__ __forceinline__ void tmem_st(uint32_t taddr, const uint32_t (&r)[16]) { tmem_st16(taddr, r); }
__device__ __forceinline__ void tmem_st(uint32_t taddr, const uint32_t (&r)[8]) { tmem_st8(taddr, r); }

// TMEM -> registers, N = 32 or 16 consecutive fp32 columns of this thread's lane
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&v)[32]) { tmem_ld32(taddr, v); }
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&v)[16]) { tmem_ld16(taddr, v); }
__device__ __forceinline__ void tmem_ld_nowait(uint32_t taddr, uint32_t (&r)[32]) { tmem_ld32_nowait(taddr, r); }
__device__ __forceinline__ void tmem_ld_nowait(uint32_t taddr, uint32_t (&r)[16]) { tmem_ld16_nowait(taddr, r); }

// Raw gate inputs of one tile held in registers by the control warp (lane owns tokens 4*lane..+3),
// loaded one tile ahead of their use so the scans never wait on global memory.
template <typename T>
struct GateRaw {
  T f[4], i[4];  // kept as loaded (no arithmetic) so the loads stay in flight until the scan
  int n_valid;
};
template <typename T>
__device__ __forceinline__ GateRaw<T> load_gate_raw(const T* ip, int64_t is, const T* fp, int64_t fs, int n_valid) {
  GateRaw<T> r;
  const int lane = threadIdx.x & 31;
  r.n_valid = n_valid;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int t = min(lane * 4 + e, n_valid - 1);  // clamp: tail tokens are masked at scan time
    r.f[e] = fp[(int64_t)t * fs];
    r.i[e] = ip[(int64_t)t * is];
  }
  return r;
}
// Control warp: gate vectors of one tile into `gb` (warp-shuffle scans, north_star item 1):
//   b = inclusive cumsum of logsigmoid(f) (fw.py:261-262), raw i, prefix max of (i - b) so that
//   m_t = b_t + max(m_prev, pm_t) (fw.py:171-184), y = (i - b) log2e, raw f, g = b_L, amax = max(i - b),
//   and the factorisation of the decay matrix used for 32x32 blocks strictly below the diagonal:
//   exp2(x_t + y_s) = exp2(x_t + ymax_u) * cf_s with cf_s = exp2(y_s - ymax_u) <= 1 (no overflow
//   because x_t + y_s <= 0 for every s <= t).  Ragged tail tokens act as logsigmoid(f) = 0, i = -inf.
// logsigmoid with the fast exp / log units (the 16-bit path tolerates 1e-6 relative error here)
__device__ __forceinline__ float logsigmoid_fast(float x) { return fminf(x, 0.f) - __logf(1.f + __expf(-fabsf(x))); }

// suffix (reverse-direction) variants of the warp scans
__device__ __forceinline__ float warp_incl_sum_dir(float v, int lane, bool rev) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float up = __shfl_up_sync(0xffffffffu, v, o), dn = __shfl_down_sync(0xffffffffu, v, o);
    if (rev ? (lane + o < 32) : (lane >= o)) v += rev ? dn : up;
  }
  return v;
}
__device__ __forceinline__ float warp_incl_max_dir(float v, int lane, bool rev) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float up = __shfl_up_sync(0xffffffffu, v, o), dn = __shfl_down_sync(0xffffffffu, v, o);
    if (rev ? (lane + o < 32) : (lane >= o)) v = fmaxf(v, rev ? dn : up);
  }
  return v;
}

// `rev`: anti-causal direction -- the cumulative sums / maxima run from the END of the tile
// (suffix scans over the memory rows), everything else is unchanged.
// `cap` > 0: the inputs are gate PRE-activations and the cell's soft cap cap * tanh(x / cap) (MatrixLSTMCell.soft_cap,
// vision_lstm2.py:714-715, 755-756) is applied here; its derivative 1 - tanh^2 goes to oDi / oDf for the backward.
template <typename T>
__device__ __noinline__ void gate_scan_regs(float* gb, const GateRaw<T>& r, bool rev, bool siging, float cap = 0.f) {
  const int lane = threadIdx.x & 31;
  float lf[4], iv[4], fv[4];
  float run = 0.f;
  if (cap > 0.f) {
    const float rc = 1.f / cap;
    float di[4], df[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float ti = tanhf(to_f32<T>(r.i[e]) * rc), tf = tanhf(to_f32<T>(r.f[e]) * rc);
      iv[e] = cap * ti;
      fv[e] = cap * tf;
      di[e] = 1.f - ti * ti;
      df[e] = 1.f - tf * tf;
    }
    reinterpret_cast<float4*>(gb + GateBuf::oDi)[lane] = make_float4(di[0], di[1], di[2], di[3]);
    reinterpret_cast<float4*>(gb + GateBuf::oDf)[lane] = make_float4(df[0], df[1], df[2], df[3]);
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      iv[e] = to_f32<T>(r.i[e]);
      fv[e] = to_f32<T>(r.f[e]);
    }
    reinterpret_cast<float4*>(gb + GateBuf::oDi)[lane] = make_float4(1.f, 1.f, 1.f, 1.f);
    reinterpret_cast<float4*>(gb + GateBuf::oDf)[lane] = make_float4(1.f, 1.f, 1.f, 1.f);
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int e = rev ? 3 - k : k;  // scan order inside the lane
    const bool ok = lane * 4 + e < r.n_valid;
    fv[e] = ok ? fv[e] : INFINITY;
    iv[e] = ok ? iv[e] : -INFINITY;
    if (siging) iv[e] = ok ? logsigmoid_fast(iv[e]) : -INFINITY;  // sigmoid input gate
    run += logsigmoid_fast(fv[e]);
    lf[e] = run;
  }
  const float incl = warp_incl_sum_dir(run, lane, rev);
  const float base = incl - run;
  float pmax = -INFINITY;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    lf[e] += base;
    pmax = fmaxf(pmax, iv[e] - lf[e]);
  }
  const float incl_max = warp_incl_max_dir(pmax, lane, rev);
  float runmax = rev ? __shfl_down_sync(0xffffffffu, incl_max, 1) : __shfl_up_sync(0xffffffffu, incl_max, 1);
  if (lane == (rev ? 31 : 0)) runmax = -INFINITY;
  // maximum of y over this lane's 32-column unit (8 lanes per unit)
  float umax = pmax;
#pragma unroll
  for (int o = 1; o < 8; o <<= 1) umax = fmaxf(umax, __shfl_xor_sync(0xffffffffu, umax, o));
  umax = fmaxf(umax * kLog2e, -1e30f);
  float pm[4], y[4], cf[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int e = rev ? 3 - k : k;
    runmax = fmaxf(runmax, iv[e] - lf[e]);
    pm[e] = runmax;
    y[e] = (iv[e] - lf[e]) * kLog2e;
    cf[e] = ex2_approx(y[e] - umax);
  }
  reinterpret_cast<float4*>(gb + GateBuf::oB)[lane] = make_float4(lf[0], lf[1], lf[2], lf[3]);
  reinterpret_cast<float4*>(gb + GateBuf::oI)[lane] = make_float4(iv[0], iv[1], iv[2], iv[3]);
  reinterpret_cast<float4*>(gb + GateBuf::oPm)[lane] = make_float4(pm[0], pm[1], pm[2], pm[3]);
  reinterpret_cast<float4*>(gb + GateBuf::oY)[lane] = make_float4(y[0], y[1], y[2], y[3]);
  reinterpret_cast<float4*>(gb + GateBuf::oF)[lane] = make_float4(fv[0], fv[1], fv[2], fv[3]);
  reinterpret_cast<float4*>(gb + GateBuf::oCf)[lane] = make_float4(cf[0], cf[1], cf[2], cf[3]);
  const float g = __shfl_sync(0xffffffffu, incl, rev ? 0 : 31);
  const float amax = warp_all_max(pmax);
  if (lane == 0) {
    gb[GateBuf::oScal + 0] = g;
    gb[GateBuf::oScal + 1] = amax;
  }
  if ((lane & 7) == 0) gb[GateBuf::oScal + 4 + (lane >> 3)] = umax;
}

// 16-bit <-> fp32 with the element type chosen at run time (the fused epilogue's x / y may be fp16 under a bf16 kernel)
__device__ __forceinline__ float2 unpack2_rt(uint32_t u, bool f16) {
  return f16 ? __half22float2(*reinterpret_cast<__half2*>(&u)) : __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
}
__device__ __forceinline__ uint32_t pack2_rt(float a, float b, bool f16) {
  return f16 ? pack2<__half>(a, b) : pack2<__nv_bfloat16>(a, b);
}

// L2 prefetch of `n_rows` rows of ROW_BYTES bytes (16-bit elements, `stride` elements apart) by one warp
template <int ROW_BYTES>
__device__ __forceinline__ void prefetch_rows_l2(const uint16_t* base, int64_t stride, int row0, int n_rows, int lane) {
  constexpr int LINES = (ROW_BYTES + 127) / 128;
  for (int r = lane; r < n_rows; r += 32) {
    const char* ptr = reinterpret_cast<const char*>(base + (int64_t)(row0 + r) * stride);
#pragma unroll
    for (int l = 0; l < LINES; ++l) asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr + l * 128));
  }
}

// Fused cell-output epilogue for one thread's slice of a staged h tile: row `row`, NC columns from `col0` of a
// [128][64]-subtiled (D = 128) or plain (D = 64 / 32) swizzled tile that already holds h rounded to the kernel dtype T.
// Each thread takes mean and centred sum of squares of ITS NC values (two passes over its own slice, no
// synchronisation); the two threads that share a row (column halves, warps w and w + 4) then exchange (mean, M2) once
// through `sstat` and a 64-thread named barrier and combine them exactly (Chan et al.: M2 = M2_a + M2_b +
// (mean_a - mean_b)^2 NC / 2) -- the same two-pass variance as the stand-alone kernel with one hand-off instead of
// three.  The skip input's row is requested from global memory before any of that (the scan warp pulled it into L2 a
// tile earlier), so its latency hides under the statistics.  The slice is then overwritten in place with
// y = (h - mean) rstd w + b + skip x in the y dtype.  (sstat is reused by the next tile only after every worker has
// passed that tile's control-warp barriers, so one barrier per tile is enough.)
// `row_var` turns the CTA's (mean, M2) over its D columns into the variance of the whole LayerNorm row (and may update
// mean): the row is these D columns (LnRowLocal), or, for rectangular heads, also the partner CTA's (tc_fw_body).
template <int D>
struct LnRowLocal {
  __device__ __forceinline__ float operator()(float&, float m2) const { return m2 * (1.f / D); }
};
template <typename T, int D, int NC, typename SwzFn, typename RowVar = LnRowLocal<D>>
__device__ __forceinline__ void ln_epilogue_slice(uint8_t* tile_slice_base, SwzFn swz, int row, int col0, int ch, int pair_bar,
                                                  float* sstat, const float* spar, const void* xrow, bool xy_f16, float ln_eps,
                                                  bool row_valid, RowVar row_var = RowVar{}) {
  // spar: [3][D] = weight, bias, skip of this head; sstat: [2][LT] means, [2][LT] centred sums of squares, by column half
  constexpr int NV = NC / 8;        // 16-byte vectors in the slice
  constexpr int XE = NV < 4 ? NV : 4;  // skip-input vectors requested up front (the rest while the first are consumed)
  const uint4* xp = (xrow && row_valid) ? reinterpret_cast<const uint4*>(xrow) : nullptr;
  uint4 xe[XE];
#pragma unroll
  for (int j = 0; j < XE; ++j) xe[j] = xp ? __ldg(xp + j) : make_uint4(0u, 0u, 0u, 0u);
  float s1 = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const uint4 u = *reinterpret_cast<const uint4*>(tile_slice_base + swz(row, col0 + 8 * j));
    const float2 a0 = unpack2<T>(u.x), a1 = unpack2<T>(u.y), a2 = unpack2<T>(u.z), a3 = unpack2<T>(u.w);
    s1 += ((a0.x + a0.y) + (a1.x + a1.y)) + ((a2.x + a2.y) + (a3.x + a3.y));
  }
  const float mean_a = s1 * (1.f / NC);
  float s2 = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const uint4 u = *reinterpret_cast<const uint4*>(tile_slice_base + swz(row, col0 + 8 * j));
    const float2 a0 = unpack2<T>(u.x), a1 = unpack2<T>(u.y), a2 = unpack2<T>(u.z), a3 = unpack2<T>(u.w);
    const float d0 = a0.x - mean_a, d1 = a0.y - mean_a, d2 = a1.x - mean_a, d3 = a1.y - mean_a, d4 = a2.x - mean_a,
                d5 = a2.y - mean_a, d6 = a3.x - mean_a, d7 = a3.y - mean_a;
    s2 += ((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3)) + ((d4 * d4 + d5 * d5) + (d6 * d6 + d7 * d7));
  }
  sstat[ch * LT + row] = mean_a;
  sstat[2 * LT + ch * LT + row] = s2;
  named_sync(pair_bar, 64);
  const float mean_b = sstat[(ch ^ 1) * LT + row], s2_b = sstat[2 * LT + (ch ^ 1) * LT + row];
  float mean = 0.5f * (mean_a + mean_b);
  const float dm = mean_a - mean_b;
  // (symmetric in a / b: both threads of the row get bit-identical statistics)
  const float rstd = rsqrtf(row_var(mean, (s2 + s2_b) + dm * dm * (0.5f * NC)) + ln_eps);
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    uint4* slot = reinterpret_cast<uint4*>(tile_slice_base + swz(row, col0 + 8 * j));
    const uint4 u = *slot;
    const float2 a[4] = {unpack2<T>(u.x), unpack2<T>(u.y), unpack2<T>(u.z), unpack2<T>(u.w)};
    uint4 xu;
    if (j < XE) xu = xe[j];
    else xu = xp ? __ldg(xp + j) : make_uint4(0u, 0u, 0u, 0u);
    const float2 x0 = unpack2_rt(xu.x, xy_f16), x1 = unpack2_rt(xu.y, xy_f16), x2 = unpack2_rt(xu.z, xy_f16), x3 = unpack2_rt(xu.w, xy_f16);
    const float xv[8] = {x0.x, x0.y, x1.x, x1.y, x2.x, x2.y, x3.x, x3.y};
    float o[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int c = col0 + 8 * j + e;
      const float hv = (e & 1) ? a[e >> 1].y : a[e >> 1].x;
      o[e] = (hv - mean) * rstd * spar[c] + spar[D + c] + spar[2 * D + c] * xv[e];
    }
    uint4 w;
    w.x = pack2_rt(o[0], o[1], xy_f16);
    w.y = pack2_rt(o[2], o[3], xy_f16);
    w.z = pack2_rt(o[4], o[5], xy_f16);
    w.w = pack2_rt(o[6], o[7], xy_f16);
    *slot = w;
  }
}

// =============================================================================================
// Forward
// =============================================================================================
struct TcFwParams {
  int B, NH, S, NT;  // NT = number of 128-token tiles
  float eps, scale;
  const void *ig, *fg;
  int64_t ig_sb, ig_sh, ig_ss, fg_sb, fg_sh, fg_ss;
  const float *c0, *n0, *m0;
  float *n_out, *m_out;
  float *c_last, *n_last, *m_last;
  int rev;           // 1: anti-causal direction (tiles walked from the end, mirrored in-tile mask)
  int sig;           // mlstm_b200_shape::siging: 1 sigmoid input gate, all max states 0; 2 the same without the
                     // normaliser (h = numerator)
  int store_states;  // 1: TMA-store the bf16 copy of C entering every tile (consumed by the backward)
  float cap;         // > 0: gate soft cap applied in the scan warp (mlstm_b200_shape::gate_soft_cap)
  // fused cell-output epilogue (mlstm_b200_fw_epilogue): the tensor map "mapH" then describes y; the plain h (if wanted)
  // is written straight from the registers
  int epi;           // 1: fused epilogue on
  int xy_f16;        // y / x element type: 1 fp16, 0 bf16
  float ln_eps;
  const float *ln_w, *ln_b, *ln_skip;  // (NH * D) fp32, each may be NULL
  const void* x;     // skip input, (B, NH, S, D) view, or NULL
  int64_t x_sb, x_sh, x_ss;
  void* h_plain;     // un-normalised h (kernel dtype), (B, NH, S, D) view, or NULL
  int64_t h_sb, h_sh, h_ss;
#ifdef MLSTM_TC_PROFILE
  long long* prof;   // per-tile phase clocks of CTA 0 (profile build only)
#endif
};

template <int D_>
struct FwSmem {
  static constexpr int D = D_;
  static constexpr int NSTAGE = 3;                   // Q / K / V ring: two tiles in flight while one is consumed
  static constexpr int kTile = Lay<D>::kTile;        // one [128][D] 16-bit tile
  static constexpr int oQ = 0;                       // [NSTAGE] Q tiles
  static constexpr int oK = oQ + NSTAGE * kTile;
  static constexpr int oV = oK + NSTAGE * kTile;
  static constexpr int oKb = oV + NSTAGE * kTile;    // abar . K
  // h staging.  kHBuf = 2 would let the TMA store of tile c drain while tile c+1 runs (128 CTAs store in
  // lock-step and a store takes up to ~3k cycles under that burst); the plumbing below supports it.
  static constexpr int kHBuf = 1;  // measured: 2 buffers at D = 64 is 1-2 us SLOWER at config 2 (40.7-42.0 vs 39.5 us)
  static constexpr int oH = oKb + kTile;
  static constexpr int oC = oH + kHBuf * kTile;      // bf16 copy of C (D x D), MMA B operand of Q [C | n]
  static constexpr int oNt = oC + Lay<D>::kState;    // second N block of that operand: column 0 = bf16 copy of n
  static constexpr int oOnes = oNt + Lay<D>::kState; // [8][128] ones, K-major: B operand of dn = Kbar^T 1
  static constexpr int oSmall = oOnes + 2048;
  // floats: gates[2], srs[2][2][LT], fused epilogue: stat[4][LT] (row partial sums), par[3][D] (weight, bias, skip)
  static constexpr int fGates = 0, fRs = 2 * GateBuf::kFloats, fStat = fRs + 4 * LT, fPar = fStat + 4 * LT,
                       kSmallFloats = fPar + 3 * D;
  static constexpr int kBytes = oSmall + kSmallFloats * 4 + 1024 /*alignment slack*/;
  // rectangular heads with the fused epilogue only (tc_fw_rect<..., EPI = true>, launched with kBytesPair): the partner
  // CTA's (mean, M2) of every row, [2 slots by tile parity][LT] float2, and one mbarrier per slot, behind everything else.
  // 2 KB more: by shared memory D = 32 still fits two CTAs per SM (2 x 112 KB), D = 64 one (212 KB).
  static constexpr int oXst = oSmall + kSmallFloats * 4, oXbar = oXst + 2 * LT * 8, kBytesPair = kBytes + 2 * LT * 8 + 16;
  static_assert(oXst % 16 == 0, "float2 slots");
  static_assert((D == 32 ? 2 : 1) * (kBytesPair + 1024 /*per-CTA reserve*/ + 256 /*static*/) <= 228 * 1024, "CTAs per SM");
  // TMEM columns.  D = 64: S double-buffered by tile parity (512 columns, one CTA per SM).  D = 32: one S
  // buffer, 256 columns, so that two CTAs share an SM (S(k+1) is issued behind the MMAs that read P(k)).
  // P (16-bit, the A operand of P V) never goes through shared memory: each thread packs its S row in
  // place -- the 16 packed columns of 32-column unit u overwrite S columns 32u .. 32u+15, which only the
  // writing warp has read -- and the MMA takes A from TMEM.
  static constexpr int kTmemCols = D == 64 ? 512 : 256;
  // Hx = Q [C | n] has D + 16 columns (column D = q . n_{k-1}); dN = Kbar^T 1 has 8 (identical) columns.
  static constexpr uint32_t cS0 = 0, cS1 = D == 64 ? 128 : 0, cHi = D == 64 ? 256 : 128, cHx = cHi + D,
                            cDC = cHx + D + 16, cDN = cDC + D;
  static_assert(cDN + 8 <= kTmemCols, "TMEM budget");
};

// ---------------------------------------------------------------------------------------------
// Stages shared by the three forward kernels (tc_fw_body, tc_fw_d128, tc_fw_wide)
// ---------------------------------------------------------------------------------------------

// Scan warp: the gate vectors of tile n go into buffer n & 1 of `gates` two tiles ahead of the workers, announced on
// bar_g[n & 1]; tiles 0 and 1 need no buffer hand-back, tile n >= 2 waits until every worker is done with tile n - 2.
// X_ROW_BYTES > 0 (fused epilogue): the skip-input rows of tile n (xbase, p.x_ss elements apart) are pulled into L2
// two tiles before the workers read them.
template <bool REV, int X_ROW_BYTES, typename T, typename MT>
__device__ __forceinline__ void fw_scan_warp(const TcFwParams& p, const T* ip, const T* fp, MT mt, float* gates,
                                             uint64_t* bar_g, const uint16_t* xbase) {
  const int lane = threadIdx.x & 31;
  auto raw_of = [&](int c) {
    const int t1 = mt(c) * LT;
    return load_gate_raw<T>(ip + (int64_t)t1 * p.ig_ss, p.ig_ss, fp + (int64_t)t1 * p.fg_ss, p.fg_ss, min(LT, p.S - t1));
  };
  GateRaw<T> raw = raw_of(0);
  for (int n = 0; n < p.NT; ++n) {
    if constexpr (X_ROW_BYTES > 0) {
      if (p.x) prefetch_rows_l2<X_ROW_BYTES>(xbase, p.x_ss, mt(n) * LT, min(LT, p.S - mt(n) * LT), lane);
    }
    if (n >= 2) named_sync(NB_C, kNbC);  // every worker is done with tile n-2: its gate buffer can be reused
    gate_scan_regs(gates + (n & 1) * GateBuf::kFloats, raw, REV, p.sig != 0, p.cap);
    __syncwarp();
    if (lane == 0) mbar_arrive(&bar_g[n & 1]);
    if (n + 1 < p.NT) raw = raw_of(n + 1);  // stays in flight until the next hand-back
  }
  for (int n = max(p.NT - 2, 0); n < p.NT; ++n) named_sync(NB_C, kNbC);  // match the workers' remaining arrivals
}

// Gate scalars of one tile for tile row `row`: g = b_L, the stabilisers m_next (end of the tile) and m_t (this row), the
// state decay gbar, and the row's b_t and i_t.  sig != 0: every max state is 0.
struct TileGates {
  float g, m_next, gbar, b_t, i_t, m_t;
};
__device__ __forceinline__ TileGates tile_gates(const float* gb, int row, float m_run, int sig) {
  const float g = gb[GateBuf::oScal], amax = gb[GateBuf::oScal + 1];
  const float m_next = sig ? 0.f : fmaxf(g + m_run, g + amax);    // fw.py:96-98
  const float gbar = __expf(g + m_run - m_next);                    // fw.py:106
  const float b_t = gb[GateBuf::oB + row], i_t = gb[GateBuf::oI + row];
  const float m_t = sig ? 0.f : b_t + fmaxf(m_run, gb[GateBuf::oPm + row]);  // fw.py:178-184
  return {g, m_next, gbar, b_t, i_t, m_t};
}

// P = S . D (causal) of tile row rb * 32 + lane over this thread's two 32-column units u = ch, ch + 2 (warp-uniform
// branches).  S is read from TMEM at tS_row (this row's lane, column 0).  sink(u, v) stores each finished unit; returns
// the row sum of P over both units.  Called by tc_fw_d128 and tc_fw_wide; tc_fw_body writes the same loop out (see there).
template <bool REV, typename Sink>
__device__ __forceinline__ float causal_p(uint32_t tS_row, const float* gb, float b_t, float m_t, float scale, int rb, int ch,
                                          int lane, Sink sink) {
  const float x_t = (b_t - m_t) * kLog2e + log2f(scale);
  const float* sy = gb + GateBuf::oY;
  const float* scf = gb + GateBuf::oCf;
  float rs = 0.f;
#pragma unroll 1
  for (int u = ch; u < 4; u += 2) {
    float v[32];
    const bool off_diag = REV ? u > rb : u < rb;  // fully unmasked 32x32 block
    if (off_diag) {  // rank-1 decay, one exp per row
      tmem_ld32(tS_row + u * 32, v);
      const float r_t = ex2_approx(x_t + gb[GateBuf::oScal + 4 + u]);
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        const float4 cf = *reinterpret_cast<const float4*>(scf + u * 32 + 4 * j4);
        v[4 * j4 + 0] *= cf.x * r_t;
        v[4 * j4 + 1] *= cf.y * r_t;
        v[4 * j4 + 2] *= cf.z * r_t;
        v[4 * j4 + 3] *= cf.w * r_t;
        rs += (v[4 * j4 + 0] + v[4 * j4 + 1]) + (v[4 * j4 + 2] + v[4 * j4 + 3]);
      }
    } else if (u == rb) {  // diagonal block: causal mask, one exp per entry
      tmem_ld32(tS_row + u * 32, v);
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        const float4 y = *reinterpret_cast<const float4*>(sy + u * 32 + 4 * j4);
        const float yy[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int j = 4 * j4 + e;
          float pv = v[j] * ex2_approx(x_t + yy[e]);
          pv = (REV ? j >= lane : j <= lane) ? pv : 0.f;
          rs += pv;
          v[j] = pv;
        }
      }
    } else {  // above the diagonal: zeros (the S MMA of every tile overwrites these columns)
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = 0.f;
    }
    sink(u, v);
  }
  return rs;
}

// One 32-column unit of P packed to 16 bits into the TMEM columns of its S unit (see FwSmem: P stays in TMEM)
template <typename T>
__device__ __forceinline__ void tmem_st_p(uint32_t taddr, const float (&v)[32]) {
  uint32_t pk[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) pk[j] = pack2<T>(v[2 * j], v[2 * j + 1]);
  tmem_st16(taddr, pk);
}

// Normaliser of row t (fw.py:197-212): bq = exp(b_t + m_{k-1} - m_t) scale scales Hinter, nmax = max(|den|, exp(-m_t)) is
// n_out, and h = (Hintra + bq Hinter) inv.  den_of(bq) returns bq (q . n_{k-1}) + the row sum of P; it runs after bq,
// so a body may wait for the TMEM loads of q . n there.
struct Normaliser {
  float bq, nmax, inv;
};
template <typename DenOf>
__device__ __forceinline__ Normaliser normaliser(const TcFwParams& p, float b_t, float m_run, float m_t, DenOf den_of) {
  const float bq = __expf(b_t + m_run - m_t) * p.scale;       // fw.py:197-198
  const float den = den_of(bq);                                // fw.py:204-206
  const float nmax = fmaxf(fabsf(den), __expf(-m_t));          // fw.py:208-210
  const float inv = p.sig == 2 ? 1.f : 1.f / (nmax + p.eps);  // siging = 2: no normaliser
  return {bq, nmax, inv};
}

// Per-channel parameters of the fused cell-output epilogue, channels col0 .. col0 + D - 1 of the layer row (spar: [3][D]
// = weight, bias, skip; a missing tensor reads as 1, 0, 0)
template <int D>
__device__ __forceinline__ void load_ln_params(const TcFwParams& p, float* spar, int col0, int tid) {
  for (int e = tid; e < D; e += kWorkers) {
    spar[e] = p.ln_w ? p.ln_w[col0 + e] : 1.f;
    spar[D + e] = p.ln_b ? p.ln_b[col0 + e] : 0.f;
    spar[2 * D + e] = p.ln_skip ? p.ln_skip[col0 + e] : 0.f;
  }
}

// VB > 1: rectangular heads, DHQK = D and DHHV = VB * D.  CTA x runs the square problem of (batch, head) x / VB on
// the D-wide column block vb = x % VB of v / h / C (see tc_fw_rect); n and m do not depend on v, so every block
// computes them and block 0 writes them.  With the fused epilogue the two blocks of a head are one {2, 1, 1} cluster
// (cluster rank = vb) and exchange the LayerNorm row statistics through distributed shared memory.
template <typename T, int D, bool REV, bool EPI, int VB>
__device__ __forceinline__ void tc_fw_body(const CUtensorMap& mapQ, const CUtensorMap& mapK, const CUtensorMap& mapV,
                                           const CUtensorMap& mapH, const CUtensorMap& mapCs, const TcFwParams& p) {
  static_assert(VB == 1 || VB == 2, "one or two column blocks");
  constexpr bool kPair = EPI && VB == 2;  // cluster launch, partner statistics
  constexpr bool kBf16 = std::is_same<T, __nv_bfloat16>::value;
  using SM = FwSmem<D>;
  using L = Lay<D>;
  constexpr int NSTAGE = SM::NSTAGE, CW = L::CW;
  TC_PROF(200, 0);  // kernel entry
  TC_PROF_CTA(0);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  float* fsm = (float*)(smem + SM::oSmall);
  uint8_t* sKb = smem + SM::oKb;
  uint8_t* sH = smem + SM::oH;
  uint8_t* sC = smem + SM::oC;
  uint8_t* sNt = smem + SM::oNt;
  uint8_t* sOnes = smem + SM::oOnes;
  __shared__ uint64_t bar_full[NSTAGE], bar_s, bar_dc, bar_h, bar_hx, bar_g[2];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // provably warp-uniform: role branches stay uniform
  const int bh = blockIdx.x / VB, vb = blockIdx.x % VB, b = bh / p.NH, hh = bh % p.NH;

  const T* ip = (const T*)p.ig + b * p.ig_sb + hh * p.ig_sh;
  const T* fp = (const T*)p.fg + b * p.fg_sb + hh * p.fg_sh;
  constexpr uint32_t kStageBytes = 3 * SM::kTile;
  // memory tile of processing tile c: the anti-causal direction walks the tiles from the end and
  // mirrors the in-tile mask / scans; no data is ever reversed (north_star item 4)
  auto mt = [&](int c) { return REV ? p.NT - 1 - c : c; };
  auto load_stage = [&](int s, int c) {
    mbar_expect_tx(&bar_full[s], kStageBytes);
    tma_load_4d(smem + SM::oQ + s * SM::kTile, &mapQ, &bar_full[s], 0, mt(c) * LT, hh, b);
    tma_load_4d(smem + SM::oK + s * SM::kTile, &mapK, &bar_full[s], 0, mt(c) * LT, hh, b);
    tma_load_4d(smem + SM::oV + s * SM::kTile, &mapV, &bar_full[s], vb * D, mt(c) * LT, hh, b);
  };
  // cold start: the first Q / K / V tiles are requested before anything else happens in the CTA.  Under
  // programmatic dependent launch every thread passes griddepcontrol.wait before ITS first global access (a no-op
  // for a normal launch), so the set-up below overlaps the tail of the previous kernel in the stream.
  if (tid == kCtlWarp * 32) {
    for (int s = 0; s < NSTAGE; ++s) mbar_init(&bar_full[s], 1);
    fence_mbar_init();
    grid_dep_wait();
    for (int s = 0; s < NSTAGE && s < p.NT; ++s) load_stage(s, s);
  }
  if (tid == 0) {
    mbar_init(&bar_s, 1);
    mbar_init(&bar_dc, 1);
    mbar_init(&bar_h, 1);
    mbar_init(&bar_hx, 1);
    mbar_init(&bar_g[0], 1);
    mbar_init(&bar_g[1], 1);
    if constexpr (kPair) {  // partner statistics of tiles of parity 0 / 1: one remote arrive per ch == 0 worker warp
      mbar_init(reinterpret_cast<uint64_t*>(smem + SM::oXbar), 4);
      mbar_init(reinterpret_cast<uint64_t*>(smem + SM::oXbar) + 1, 4);
    }
    fence_mbar_init();
  }
  if (warp == kCtlWarp) {
    tmem_alloc<SM::kTmemCols>(&tmem_base_s);
    if (lane == 0) {
      prefetch_tmap(&mapQ); prefetch_tmap(&mapK); prefetch_tmap(&mapV); prefetch_tmap(&mapH); prefetch_tmap(&mapCs);
    }
  }
  grid_dep_wait();
  grid_dep_launch();
  // worker-side state: fp32 master copy of C in the registers of lanes < 16 of the worker warps:
  // row d = 16*rb + lane (M=64 TMEM layout; D = 32 has 32 real rows, warps rb < 2), columns CW*ch .. CW*ch+CW-1;
  // the ch == 0 owner of a row also keeps n[d] (fp32) and its 16-bit operand copy in sNt(d, 0)
  const int rb = warp & 3, ch = (warp >> 2) & 1;
  const int row = rb * 32 + lane;  // tile row == TMEM lane of this thread
  const uint32_t lane_base = (uint32_t)(rb * 32) << 16;
  const int drow = rb * 16 + (lane & 15);
  const bool owns_c = warp < kCtlWarp && lane < 16 && rb * 16 < D;
  float Creg[CW];
  float n_reg = 0.f;
#pragma unroll
  for (int j = 0; j < CW; ++j) Creg[j] = 0.f;
  if (warp < kCtlWarp) {
    if (p.c0 && owns_c) {
      const float* src = p.c0 + ((int64_t)bh * D + drow) * (VB * D) + vb * D + ch * CW;
#pragma unroll
      for (int j = 0; j < CW; ++j) Creg[j] = src[j];
    }
    if (owns_c) store_cols<T, D>(sC, drow, ch * CW, Creg);
    for (int e = tid; e < L::kState / 16; e += kWorkers) reinterpret_cast<uint4*>(sNt)[e] = make_uint4(0, 0, 0, 0);
    {
      const uint32_t one2 = pack2<T>(1.f, 1.f);
      for (int e = tid; e < 2048 / 16; e += kWorkers) reinterpret_cast<uint4*>(sOnes)[e] = make_uint4(one2, one2, one2, one2);
    }
    if (EPI) load_ln_params<D>(p, fsm + SM::fPar, hh * (VB * D) + vb * D, tid);  // this head's column block
    named_sync(NB_PAIR0, kWorkers);  // sNt zeroed before the owners write column 0
    if (owns_c && ch == 0) {
      n_reg = p.n0 ? p.n0[(int64_t)bh * D + drow] : 0.f;
      *reinterpret_cast<T*>(sNt + L::swz(drow, 0)) = from_f32<T>(n_reg);
    }
    fence_proxy_async_smem();
  }
  if (warp == kScanWarp) {  // cold start: pull the first tile's gate rows towards L2 / L1 while the CTA sets up
    const int t1 = mt(0) * LT, nv = min(LT, p.S - t1);
    for (int e = lane; e < nv; e += 32) {
      asm volatile("prefetch.global.L1 [%0];" ::"l"(ip + (int64_t)(t1 + e) * p.ig_ss));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(fp + (int64_t)(t1 + e) * p.fg_ss));
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  if constexpr (kPair) cluster_sync();  // the partner's mbarriers are initialised before the first remote arrive
  const uint32_t tmem = tmem_base_s;
  const uint32_t tS0 = tmem + SM::cS0, tS1 = tmem + SM::cS1, tHi = tmem + SM::cHi, tHx = tmem + SM::cHx, tDC = tmem + SM::cDC,
                 tDN = tmem + SM::cDN;

  if (warp == kCtlWarp) {
    // =========================== control warp ===================================================
    constexpr uint32_t id_s = umma_idesc(128, 128, false, false, kBf16);
    constexpr uint32_t id_dc = umma_idesc(64, D, true, true, kBf16);
    constexpr uint32_t id_h = umma_idesc(128, D, false, true, kBf16);
    constexpr uint32_t id_hx = umma_idesc(128, D + 16, false, true, kBf16);  // Q [C | n]
    constexpr uint32_t id_dn = umma_idesc(64, 8, true, false, kBf16);        // Kbar^T 1
    const uint64_t dOnes = umma_smem_desc(smem_u32(sOnes), 0, 1024);
    const uint64_t dKb = L::desc(smem_u32(sKb), D == 64 ? SM::kTile : 0);  // D = 32: rows 32-63 of the M = 64 MMA re-read the block
    const uint64_t dC = L::desc(smem_u32(sC), L::kState);
    // Every shared-memory descriptor is provably warp-uniform (stage-0 descriptor + stage index * tile bytes;
    // the TMEM parity is a compile-time constant of the two-tile unrolled body), so the tcgen05.mma operands
    // live in uniform registers instead of going through a per-instruction R2UR waterfall.
    const uint64_t dQ0 = L::desc(smem_u32(smem + SM::oQ), 0);
    const uint64_t dK0 = L::desc(smem_u32(smem + SM::oK), 0);
    const uint64_t dV0 = L::desc(smem_u32(smem + SM::oV), SM::kTile);
    auto issue_s = [&](int c, auto PAR) {  // S(c) = Q K^T into the TMEM buffer of the tile's parity
      constexpr int par = decltype(PAR)::value;
      const int s = c % NSTAGE;
      mbar_wait(&bar_full[s], (c / NSTAGE) & 1, 1);
      tc_fence_after_sync();
      const uint64_t dQ = umma_desc_advance(dQ0, s * SM::kTile), dK = umma_desc_advance(dK0, s * SM::kTile);
      const uint32_t tS = par ? tS1 : tS0;
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        umma_f16(tS, umma_desc_advance(dQ, kk * 32), umma_desc_advance(dK, kk * 32), id_s, kk > 0);
      umma_commit(&bar_s);
    };
    if (lane == 0 && p.store_states) {  // state entering tile 0 (bf16 operand copy) -> c_states[b, h, 0]
      tma_store_4d(&mapCs, sC, 0, mt(0) * (VB * D) + vb * D, hh, b);
      tma_store_commit();
    }
    __syncwarp();
    if (elect_one()) issue_s(0, std::integral_constant<int, 0>{});
    __syncwarp();

    auto tile_body = [&](int c, auto PAR) {
      constexpr int par = decltype(PAR)::value;
      const int s = c % NSTAGE;
      const uint64_t dQ = umma_desc_advance(dQ0, s * SM::kTile), dV = umma_desc_advance(dV0, s * SM::kTile);
      TC_PROF(c, 9);
      // Hinter = Q [C_{k-1} | n_{k-1}] (column D is q . n_{k-1}) depends on nothing this tile computes: the state
      // copies were written before the previous tile's NB_C and its Q tile has landed (S(c) waited for it), so
      // it runs under the workers' P phase instead of behind P V on the S -> P -> PV -> epilogue chain.
      if (elect_one()) {  // elect.sync lets ptxas emit straight-line UTCHMMA (no per-instruction thread loop)
        tc_fence_after_sync();
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk)
          umma_f16(tHx, umma_desc_advance(dQ, kk * 32), umma_desc_advance(dC, kk * L::kAdvMN), id_hx, kk > 0);
        umma_commit(&bar_hx);
      }
      __syncwarp();
      named_sync(NB_B, kNbAB);  // P(c) written
      if (lane == 0) {
        // the stores that read the buffers rewritten after bar_h -- sC (c_states) and this tile's h staging buffer --
        // are done; with two h buffers the newest group (h of the previous tile) may still be in flight
        tma_store_wait_read<SM::kHBuf - 1>();
        TC_PROF(c, 10);
      }
      __syncwarp();
      if (elect_one()) {
        tc_fence_after_sync();
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // Hintra = P V, A = P from TMEM (packed inside the S columns)
          umma_f16_ts(tHi, (par ? tS1 : tS0) + 32 * (kk / 2) + 8 * (kk % 2), umma_desc_advance(dV, kk * L::kAdvMN), id_h, kk > 0);
        umma_commit(&bar_h);
      }
      __syncwarp();
      TC_PROF(c, 11);
      named_sync(NB_A, kNbAB);  // Kbar(c) written
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // dC = Kbar^T V
          umma_f16(tDC, umma_desc_advance(dKb, kk * L::kAdvMN), umma_desc_advance(dV, kk * L::kAdvMN), id_dc, kk > 0);
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // dn = Kbar^T 1 (column sums on the tensor pipe)
          umma_f16(tDN, umma_desc_advance(dKb, kk * L::kAdvMN), umma_desc_advance(dOnes, (kk / 4) * 1024 + (kk % 4) * 32), id_dn,
                   kk > 0);
        umma_commit(&bar_dc);
        if (c + 1 < p.NT) issue_s(c + 1, std::integral_constant<int, par ^ 1>{});  // next tile's S, other TMEM buffer
      }
      __syncwarp();
      TC_PROF(c, 13);
      named_sync(NB_C, kNbC);  // h staged, C_k written: every worker is done with this tile
      if (lane == 0) {
        TC_PROF(c, 14);
        if (p.store_states && c + 1 < p.NT) {  // state entering tile c+1; its own, OLDER group than h(c): see the wait above
          tma_store_4d(&mapCs, sC, 0, mt(c + 1) * (VB * D) + vb * D, hh, b);
          tma_store_commit();
        }
        tma_store_4d(&mapH, sH + (SM::kHBuf == 2 ? (c & 1) * SM::kTile : 0), vb * D, mt(c) * LT, hh, b);
        tma_store_commit();
        if (c + NSTAGE < p.NT) load_stage(s, c + NSTAGE);
        TC_PROF(c, 15);
      }
      __syncwarp();
    };
    for (int c = 0; c < p.NT; c += 2) {
      tile_body(c, std::integral_constant<int, 0>{});
      if (c + 1 < p.NT) tile_body(c + 1, std::integral_constant<int, 1>{});
    }
    if (lane == 0) tma_store_wait_all<0>();
  } else if (warp == kScanWarp) {
    fw_scan_warp<REV, EPI ? D * 2 : 0>(p, ip, fp, mt, fsm + SM::fGates, bar_g,
                                       p.x ? (const uint16_t*)p.x + b * p.x_sb + hh * p.x_sh + vb * D : nullptr);
  } else {
    // =========================== worker warps ===================================================
    float m_run = p.m0 ? p.m0[bh] : 0.f;
    for (int c = 0; c < p.NT; ++c) {
      const int s = c % NSTAGE, pb = c & 1;
      const uint32_t par_full = (c / NSTAGE) & 1, par = c & 1;
      const uint8_t* sQ = smem + SM::oQ + s * SM::kTile;
      const uint8_t* sK = smem + SM::oK + s * SM::kTile;
      const float* gb = fsm + SM::fGates + pb * GateBuf::kFloats;
      float* srs = fsm + SM::fRs + pb * 2 * LT;
      const int t0 = mt(c) * LT;
      const int n_valid = min(LT, p.S - t0);
      const uint32_t tS = (c & 1) ? tS1 : tS0;

      TC_PROF(c, 0);
      mbar_wait(&bar_g[pb], (c >> 1) & 1, 2);
      const auto [g, m_next, gbar, b_t, i_t, m_t] = tile_gates(gb, row, m_run, p.sig);
      TC_PROF(c, 1);
      // ---- P = S . D (causal), row sums; P packed into the S columns ----------------------------
      mbar_wait(&bar_s, par, 5);
      tc_fence_after_sync();
      TC_PROF(c, 2);
      {
        const float x_t = (b_t - m_t) * kLog2e + log2f(p.scale);
        const float* sy = gb + GateBuf::oY;
        const float* scf = gb + GateBuf::oCf;
        float rs = 0.f;
#pragma unroll 1
        // causal_p's loop, written out here: called, it changes this kernel's register allocation and costs the (64, 128)
        // forward 0.4 % at S = 6400 (B200); keep the two copies in step
        for (int u = ch; u < 4; u += 2) {  // this thread's two 32-column units (warp-uniform branches)
          float v[32];
          const bool off_diag = REV ? u > rb : u < rb;  // fully unmasked 32x32 block
          if (off_diag) {  // rank-1 decay, one exp per row
            tmem_ld32(tS + lane_base + u * 32, v);
            const float r_t = ex2_approx(x_t + gb[GateBuf::oScal + 4 + u]);
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 cf = *reinterpret_cast<const float4*>(scf + u * 32 + 4 * j4);
              v[4 * j4 + 0] *= cf.x * r_t;
              v[4 * j4 + 1] *= cf.y * r_t;
              v[4 * j4 + 2] *= cf.z * r_t;
              v[4 * j4 + 3] *= cf.w * r_t;
              rs += (v[4 * j4 + 0] + v[4 * j4 + 1]) + (v[4 * j4 + 2] + v[4 * j4 + 3]);
            }
          } else if (u == rb) {  // diagonal block: causal mask, one exp per entry
            tmem_ld32(tS + lane_base + u * 32, v);
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              const float4 y = *reinterpret_cast<const float4*>(sy + u * 32 + 4 * j4);
              const float yy[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int j = 4 * j4 + e;
                float pv = v[j] * ex2_approx(x_t + yy[e]);
                pv = (REV ? j >= lane : j <= lane) ? pv : 0.f;
                rs += pv;
                v[j] = pv;
              }
            }
          } else {  // above the diagonal: zeros (the S MMA of every tile overwrites these columns)
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0.f;
          }
          uint32_t pk[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) pk[j] = pack2<T>(v[2 * j], v[2 * j + 1]);
          tmem_st16(tS + lane_base + u * 32, pk);
        }
        srs[ch * LT + row] = rs;
      }
      TC_PROF(c, 3);
      tmem_st_wait();
      TC_PROF(c, 4);
      tc_fence_before_sync();
      named_arrive(NB_B, kNbAB);
      TC_PROF(c, 5);
      // (the loads and n_{k-1} are only needed from here on: their waits stay off the S -> P -> PV chain)
      mbar_wait(&bar_full[s], par_full, 3);
      // ---- Kbar = abar . K (this thread: row, CW columns); overlaps the H MMAs ---------------------------
      {
        const float ab = __expf(g - b_t + i_t - m_next);  // fw.py:102 (exp(-inf) = 0 for tail tokens)
        float kb[CW];
#pragma unroll
        for (int j = 0; j < CW / 8; ++j) {
          uint4 u = *reinterpret_cast<const uint4*>(sK + L::swz(row, ch * CW + 8 * j));
          float2 a0 = unpack2<T>(u.x), a1 = unpack2<T>(u.y), a2 = unpack2<T>(u.z), a3 = unpack2<T>(u.w);
          kb[8 * j + 0] = a0.x * ab; kb[8 * j + 1] = a0.y * ab; kb[8 * j + 2] = a1.x * ab; kb[8 * j + 3] = a1.y * ab;
          kb[8 * j + 4] = a2.x * ab; kb[8 * j + 5] = a2.y * ab; kb[8 * j + 6] = a3.x * ab; kb[8 * j + 7] = a3.y * ab;
        }
        store_cols<T, D>(sKb, row, ch * CW, kb);
        fence_proxy_async_smem();
        named_arrive(NB_A, kNbAB);
      }
      TC_PROF(c, 6);
      // ---- epilogue -----------------------------------------------------------------------------------
      mbar_wait(&bar_hx, par, 9);
      mbar_wait(&bar_h, par, 7);
      tc_fence_after_sync();
      TC_PROF(c, 7);
      {
        uint32_t hi[CW], hx[CW], qn_u;
        tmem_ld_nowait(tHi + lane_base + ch * CW, hi);
        tmem_ld_nowait(tHx + lane_base + ch * CW, hx);
        tmem_ld1_nowait(tHx + lane_base + D, qn_u);  // q . n_{k-1}
        const auto [bq, nmax, inv] = normaliser(p, b_t, m_run, m_t, [&](float bq_t) {
          const float rs = srs[row] + srs[LT + row];
          tmem_ld_wait();
          return bq_t * __uint_as_float(qn_u) + rs;
        });
        float o[CW];
#pragma unroll
        for (int j = 0; j < CW; ++j) o[j] = (__uint_as_float(hi[j]) + bq * __uint_as_float(hx[j])) * inv;  // fw.py:200-212
        uint8_t* sHc = sH + (SM::kHBuf == 2 ? (c & 1) * SM::kTile : 0);
        store_cols<T, D>(sHc, row, ch * CW, o);
        if (ch == 0 && row < n_valid && vb == 0) {
          p.n_out[(int64_t)bh * p.S + t0 + row] = nmax;
          p.m_out[(int64_t)bh * p.S + t0 + row] = m_t;
        }
        if (EPI) {
          // fused cell output (mlstm_b200_fw_epilogue): the un-normalised row goes out from the staged copy (training:
          // the LayerNorm backward needs it), then the staged slice becomes y = LN(h) w + b + skip x
          const int64_t tok = (int64_t)(t0 + row);
          const int col = vb * D + ch * CW;  // first column of this thread's slice in the DHHV-wide row
          if (p.h_plain && row < n_valid) {
            uint4* dst = reinterpret_cast<uint4*>((T*)p.h_plain + b * p.h_sb + hh * p.h_sh + tok * p.h_ss + col);
#pragma unroll
            for (int j = 0; j < CW / 8; ++j) dst[j] = *reinterpret_cast<const uint4*>(sHc + L::swz(row, ch * CW + 8 * j));
          }
          const void* xrow = p.x ? (const void*)((const uint16_t*)p.x + b * p.x_sb + hh * p.x_sh + tok * p.x_ss + col) : nullptr;
          if constexpr (!kPair) {
            ln_epilogue_slice<T, D, CW>(sHc, [](int r, int cc) { return L::swz(r, cc); }, row, ch * CW, ch, NB_PAIR0 + rb,
                                        fsm + SM::fStat, fsm + SM::fPar, xrow, p.xy_f16 != 0, p.ln_eps, row < n_valid);
          } else {
            // The row's other D columns are in the partner CTA (cluster rank vb ^ 1).  The ch == 0 thread of every row
            // -- every row, valid or not, so that each tile sees its 4 arrivals -- writes this block's (mean, M2) into
            // the partner's slot of the tile's parity, and each of the 4 ch == 0 warps then arrives once on the partner's
            // mbarrier of that slot; both threads of the row wait for the partner's arrivals on the local one and combine
            // the two blocks in block order (bit-identical mean and rstd in both CTAs), exactly as the in-CTA halves.
            // Two slots are enough: the partner writes tile c + 2 into this slot only after it has received our tile
            // c + 1 statistics, which the ch == 0 thread sends after this tile's pair barrier of tile c + 1 -- that is,
            // after both threads of the row have read the slot for tile c.  The same ordering keeps each mbarrier at
            // most one phase ahead of its waiters, so the parity wait cannot skip a phase.
            auto pair_var = [&](float& mean, float m2) {
              float2* xst = reinterpret_cast<float2*>(smem + SM::oXst) + (c & 1) * LT;
              uint64_t* xbar = reinterpret_cast<uint64_t*>(smem + SM::oXbar) + (c & 1);
              if (ch == 0) {  // warp-uniform
                st_cluster_f2(cluster_map(xst + row, vb ^ 1), mean, m2);
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(cluster_map(xbar, vb ^ 1));
              }
              mbar_wait_cluster(xbar, (c >> 1) & 1);
              const float2 o = xst[row];
              const float mean0 = vb ? o.x : mean, mean1 = vb ? mean : o.x, m2_0 = vb ? o.y : m2, m2_1 = vb ? m2 : o.y;
              const float dmb = mean0 - mean1;
              mean = 0.5f * (mean0 + mean1);
              return ((m2_0 + m2_1) + dmb * dmb * (0.5f * D)) * (1.f / (2 * D));
            };
            ln_epilogue_slice<T, D, CW>(sHc, [](int r, int cc) { return L::swz(r, cc); }, row, ch * CW, ch, NB_PAIR0 + rb,
                                        fsm + SM::fStat, fsm + SM::fPar, xrow, p.xy_f16 != 0, p.ln_eps, row < n_valid, pair_var);
          }
        }
      }
      // ---- state update C_k = gbar C_{k-1} + dC; n_k ---------------------------------------------------
      mbar_wait(&bar_dc, par, 6);
      tc_fence_after_sync();
      {
        uint32_t v[CW], dn_u;
        tmem_ld_nowait(tDC + lane_base + ch * CW, v);  // M=64 layout: lanes 0-15 of each quadrant hold rows
        tmem_ld1_nowait(tDN + lane_base, dn_u);
        tmem_ld_wait();
        if (owns_c) {
#pragma unroll
          for (int j = 0; j < CW; ++j) Creg[j] = gbar * Creg[j] + __uint_as_float(v[j]);
          store_cols<T, D>(sC, drow, ch * CW, Creg);  // Q [C | n]_{k-1} (bar_hx) has finished reading the old copies
          if (ch == 0) {  // n_k = gbar n_{k-1} + column sums of Kbar (fw.py:116)
            n_reg = gbar * n_reg + __uint_as_float(dn_u);
            *reinterpret_cast<T*>(sNt + L::swz(drow, 0)) = from_f32<T>(n_reg);
          }
        }
      }
      fence_proxy_async_smem();
      tc_fence_before_sync();
      named_arrive(NB_C, kNbC);
      TC_PROF(c, 8);
      m_run = m_next;
    }
    // final states (fw.py:302-309)
    if (p.c_last) {
      if (owns_c) {
        float* dst = p.c_last + ((int64_t)bh * D + drow) * (VB * D) + vb * D + ch * CW;
#pragma unroll
        for (int j = 0; j < CW; ++j) dst[j] = Creg[j];
      }
      if (owns_c && ch == 0 && vb == 0) p.n_last[(int64_t)bh * D + drow] = n_reg;
      if (tid == 0 && vb == 0) p.m_last[bh] = m_run;
    }
  }
  TC_PROF(200, 1);  // this role is done
  tc_fence_before_sync();
  __syncthreads();
  TC_PROF(200, 2);
  TC_PROF_CTA(1);
  if (warp == kCtlWarp) tmem_dealloc<SM::kTmemCols>(tmem);
  if constexpr (kPair) cluster_sync();  // neither CTA exits while its partner may still write into its shared memory
}

template <typename T, int D, bool REV, bool EPI>
__global__ void __launch_bounds__(kTcThreads, D == 32 ? 2 : 1)
tc_fw(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
          const __grid_constant__ CUtensorMap mapV, const __grid_constant__ CUtensorMap mapH,
          const __grid_constant__ CUtensorMap mapCs, TcFwParams p) {
  tc_fw_body<T, D, REV, EPI, 1>(mapQ, mapK, mapV, mapH, mapCs, p);
}

// Rectangular heads DHQK = D, DHHV = 2 D: the two square column-block problems of every (batch, head) in one launch
// (grid 2 B NH, the two blocks of a head on adjacent CTAs so that their Q / K reads meet in L2).  Shared memory, TMEM
// columns and CTAs per SM are those of tc_fw<T, D>; mapV / mapH are DHHV wide with D-wide boxes, and mapCs is the
// block layout of make_states_map_blocks (the state entering tile c, column block vb, at rows (2 c + vb) D).
// EPI: fused cell-output epilogue, launched as {2, 1, 1} clusters (run_fw) with FwSmem<D>::kBytesPair.
template <typename T, int D, bool REV, bool EPI>
__global__ void __launch_bounds__(kTcThreads, D == 32 ? 2 : 1)
tc_fw_rect(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
           const __grid_constant__ CUtensorMap mapV, const __grid_constant__ CUtensorMap mapH,
           const __grid_constant__ CUtensorMap mapCs, TcFwParams p) {
  tc_fw_body<T, D, REV, EPI, 2>(mapQ, mapK, mapV, mapH, mapCs, p);
}

// =============================================================================================
// Forward, head dim 128 (640-base384.yaml: NH=6, DH=128; the inference config of BASELINE.json).
// Same algorithm, warp roles and shared stages (fw_scan_warp, tile_gates, normaliser) as tc_fw_body;
// differences: every Q/K/V/H/C tile is two [128][64]
// swizzled sub-tiles (column halves), dC = Kbar^T V is M128 N128 so C lives in the plain TMEM
// lane == row layout (every worker thread owns C[row][64 columns] in 64 registers), shared memory
// (192 KB of tiles) leaves room for ONE Q/K/V stage and S is single-buffered in TMEM (4 x 128 columns).
// =============================================================================================
struct FwSmem128 {
  static constexpr int D = 128;
  static constexpr int kTile = LT * 128;      // one [128][64] sub-tile
  static constexpr int oQ = 0, oK = 2 * kTile, oV = 4 * kTile;
  static constexpr int oKb = 6 * kTile;       // abar . K
  static constexpr int oP = 8 * kTile;        // P (two K-halves); the h staging tile aliases it
  static constexpr int oC = 10 * kTile;       // bf16 copy of C: [128 dqk rows][128 dv cols]
  static constexpr int oSmall = 12 * kTile;
  // floats: gates[2], srs[2][2][LT], sqn[2][2][LT], npart[2][4][D], sN[2][D], fused epilogue: stat[4][LT], par[3][D]
  static constexpr int fGates = 0, fRs = 2 * GateBuf::kFloats, fQn = fRs + 4 * LT, fNp = fQn + 4 * LT,
                       fN = fNp + 8 * D, fStat = fN + 2 * D, fPar = fStat + 4 * LT, kSmallFloats = fPar + 3 * D;
  static constexpr int kBytes = oSmall + kSmallFloats * 4 + 1024;
  static constexpr uint32_t kLoadBytes = 6 * kTile;
};

// ---- pieces of the M128-layout forwards (tc_fw_d128, tc_fw_wide): C in the plain TMEM lane == row layout, every worker
// thread keeps 64 fp32 columns of one C row in registers (Creg) ---------------------------------------------------------

// Set-up: thread 0 initialises the mbarriers (bar_n takes n_arrivals per phase, the others one), the control warp
// allocates the 512 TMEM columns and prefetches the four tensor maps.
__device__ __forceinline__ void fw128_prologue(int warp, uint64_t& bar_full, uint64_t& bar_s, uint64_t& bar_dc, uint64_t& bar_h,
                                               uint64_t (&bar_g)[2], uint64_t& bar_n, uint32_t n_arrivals, uint32_t& tmem_base_s,
                                               const CUtensorMap& m0, const CUtensorMap& m1, const CUtensorMap& m2,
                                               const CUtensorMap& m3) {
  if (threadIdx.x == 0) {
    mbar_init(&bar_full, 1);
    mbar_init(&bar_s, 1);
    mbar_init(&bar_dc, 1);
    mbar_init(&bar_h, 1);
    mbar_init(&bar_g[0], 1);
    mbar_init(&bar_g[1], 1);
    mbar_init(&bar_n, n_arrivals);
    fence_mbar_init();
  }
  if (warp == kCtlWarp) {
    tmem_alloc<512>(&tmem_base_s);
    if ((threadIdx.x & 31) == 0) {
      prefetch_tmap(&m0); prefetch_tmap(&m1); prefetch_tmap(&m2); prefetch_tmap(&m3);
    }
  }
}

// C_0: Creg = the row at c0 + off (c0 NULL: Creg keeps its zeros), and its 16-bit operand copy into row srow, columns
// col0 .. col0 + 63 of sC
template <typename T>
__device__ __forceinline__ void fw128_load_c0(float (&Creg)[64], const float* c0, int64_t off, uint8_t* sC, int srow, int col0) {
  if (c0) {
    const float* src = c0 + off;
#pragma unroll
    for (int j = 0; j < 64; ++j) Creg[j] = src[j];
  }
#pragma unroll
  for (int hf = 0; hf < 2; ++hf) {
    float t32[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) t32[j] = Creg[hf * 32 + j];
    store_row32<T>(sC, srow, col0 + hf * 32, t32);
  }
}

// C_k = gbar C_{k-1} + dC (dC: this thread's 64 columns in TMEM from tDC_row) and its 16-bit operand copy, placed as in
// fw128_load_c0
template <typename T>
__device__ __forceinline__ void fw128_update_c(float (&Creg)[64], float gbar, uint32_t tDC_row, uint8_t* sC, int srow, int col0) {
#pragma unroll
  for (int hf = 0; hf < 2; ++hf) {
    float v[32], t32[32];
    tmem_ld32(tDC_row + hf * 32, v);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      Creg[hf * 32 + j] = gbar * Creg[hf * 32 + j] + v[j];
      t32[j] = Creg[hf * 32 + j];
    }
    store_row32<T>(sC, srow, col0 + hf * 32, t32);  // Q C_{k-1} (bar_h) has finished reading the old copy
  }
}

template <typename T, bool REV, bool EPI>
__global__ void __launch_bounds__(kTcThreads, 1)
tc_fw_d128(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
           const __grid_constant__ CUtensorMap mapV, const __grid_constant__ CUtensorMap mapH,
           const __grid_constant__ CUtensorMap mapCs, TcFwParams p) {
  constexpr int D = 128;
  constexpr bool kBf16 = std::is_same<T, __nv_bfloat16>::value;
  using SM = FwSmem128;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float* fsm = (float*)(smem + SM::oSmall);
  uint8_t* sQ = smem + SM::oQ;
  uint8_t* sK = smem + SM::oK;
  uint8_t* sV = smem + SM::oV;
  uint8_t* sKb = smem + SM::oKb;
  uint8_t* sP = smem + SM::oP;
  uint8_t* sH = sP;
  uint8_t* sC = smem + SM::oC;
  __shared__ uint64_t bar_full, bar_s, bar_dc, bar_h, bar_g[2], bar_n;
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int bh = blockIdx.x, b = bh / p.NH, hh = bh % p.NH;

  fw128_prologue(warp, bar_full, bar_s, bar_dc, bar_h, bar_g, bar_n, D, tmem_base_s, mapQ, mapK, mapV, mapH);
  const int rb = warp & 3, ch = (warp >> 2) & 1;
  const int row = rb * 32 + lane;  // tile row == TMEM lane; also the dqk row of C this thread owns
  const uint32_t lane_base = (uint32_t)(rb * 32) << 16;
  float Creg[64];                  // C[row][64*ch .. 64*ch+63], fp32 master copy
#pragma unroll
  for (int j = 0; j < 64; ++j) Creg[j] = 0.f;
  if (warp < kCtlWarp) {
    fw128_load_c0<T>(Creg, p.c0, ((int64_t)bh * D + row) * D + ch * 64, sC, row, ch * 64);
    if (tid < D) fsm[SM::fN + tid] = p.n0 ? p.n0[(int64_t)bh * D + tid] : 0.f;
    if (EPI) load_ln_params<D>(p, fsm + SM::fPar, hh * D, tid);  // this head
    fence_proxy_async_smem();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_s;
  const uint32_t tS = tmem, tHi = tmem + 128, tHx = tmem + 256, tDC = tmem + 384;

  const T* ip = (const T*)p.ig + b * p.ig_sb + hh * p.ig_sh;
  const T* fp = (const T*)p.fg + b * p.fg_sb + hh * p.fg_sh;
  auto mt = [&](int c) { return REV ? p.NT - 1 - c : c; };

  if (warp == kCtlWarp) {
    // =========================== control warp ===================================================
    auto load_tile = [&](int c) {
      mbar_expect_tx(&bar_full, SM::kLoadBytes);
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        tma_load_4d(sQ + hf * SM::kTile, &mapQ, &bar_full, hf * 64, mt(c) * LT, hh, b);
        tma_load_4d(sK + hf * SM::kTile, &mapK, &bar_full, hf * 64, mt(c) * LT, hh, b);
        tma_load_4d(sV + hf * SM::kTile, &mapV, &bar_full, hf * 64, mt(c) * LT, hh, b);
      }
    };
    // One shared-memory stage only (192 KB of tiles): the refill of tile c+1 can start when every MMA of tile c has
    // read Q / K / V, so its latency is exposed.  The tiles are therefore pulled into L2 two tiles ahead (no shared
    // memory needed), which turns the refill into an L2 hit.
    auto prefetch_tile = [&](int c) {
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        tma_prefetch_4d(&mapQ, hf * 64, mt(c) * LT, hh, b);
        tma_prefetch_4d(&mapK, hf * 64, mt(c) * LT, hh, b);
        tma_prefetch_4d(&mapV, hf * 64, mt(c) * LT, hh, b);
      }
    };
    constexpr uint32_t id_kk = umma_idesc(128, 128, false, false, kBf16);  // A K-major, B K-major
    constexpr uint32_t id_mm = umma_idesc(128, 128, true, true, kBf16);    // A MN-major, B MN-major
    constexpr uint32_t id_km = umma_idesc(128, 128, false, true, kBf16);   // A K-major, B MN-major
    const uint64_t dQ = umma_smem_desc(smem_u32(sQ), 0, 1024), dK = umma_smem_desc(smem_u32(sK), 0, 1024);
    const uint64_t dV = umma_smem_desc(smem_u32(sV), SM::kTile, 1024);
    const uint64_t dKb = umma_smem_desc(smem_u32(sKb), SM::kTile, 1024);
    const uint64_t dP = umma_smem_desc(smem_u32(sP), 0, 1024);
    const uint64_t dC = umma_smem_desc(smem_u32(sC), SM::kTile, 1024);
    auto issue_s = [&](int c) {  // S(c) = Q K^T
      mbar_wait(&bar_full, c & 1, 1);
      tc_fence_after_sync();
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        umma_f16(tS, umma_desc_advance(dQ, (kk / 4) * SM::kTile + (kk % 4) * 32),
                 umma_desc_advance(dK, (kk / 4) * SM::kTile + (kk % 4) * 32), id_kk, kk > 0);
      umma_commit(&bar_s);
    };
    // State entering tile c, for the backward: the 16-bit operand copy of C is stored as its four 64 x 64 blocks
    // (block = 2 * (dqk half) + (dv half)), 256 rows of 64 columns per tile, which is what the four head-dim-64
    // block problems of the backward load (bw_by_blocks).  sC holds two [128][64] column halves; a block is
    // 64 consecutive rows (8 KB) of one half.
    auto store_state = [&](int c) {
#pragma unroll
      for (int blk = 0; blk < 4; ++blk)
        tma_store_4d(&mapCs, sC + (blk & 1) * SM::kTile + (blk >> 1) * 8192, 0, mt(c) * 256 + blk * 64, hh, b);
    };
    if (lane == 0) {
      if (p.store_states) {
        store_state(0);
        tma_store_commit();
      }
      load_tile(0);
      if (p.NT > 1) prefetch_tile(1);
    }
    __syncwarp();
    if (elect_one()) issue_s(0);
    __syncwarp();
    for (int c = 0; c < p.NT; ++c) {
      const uint32_t par = c & 1;
      if (lane == 0 && c + 2 < p.NT) prefetch_tile(c + 2);
      named_sync(NB_B, kNbAB);  // P(c) written
      if (c == 0 && lane == 0) tma_store_wait_read<0>();  // the initial-state store has read sC (rewritten after bar_h)
      __syncwarp();
      if (elect_one()) {
        tc_fence_after_sync();
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // Hintra = P V
          umma_f16(tHi, umma_desc_advance(dP, (kk / 4) * SM::kTile + (kk % 4) * 32), umma_desc_advance(dV, kk * 2048), id_km,
                   kk > 0);
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk)  // Hinter = Q C_{k-1}
          umma_f16(tHx, umma_desc_advance(dQ, (kk / 4) * SM::kTile + (kk % 4) * 32), umma_desc_advance(dC, kk * 2048), id_km,
                   kk > 0);
        umma_commit(&bar_h);
      }
      __syncwarp();
      named_sync(NB_A, kNbAB);  // Kbar(c) written
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // dC = Kbar^T V
          umma_f16(tDC, umma_desc_advance(dKb, kk * 2048), umma_desc_advance(dV, kk * 2048), id_mm, kk > 0);
        umma_commit(&bar_dc);
        mbar_wait(&bar_h, par, 8);   // every MMA of this tile has read Q/K/V: refill the single stage
        mbar_wait(&bar_dc, par, 9);
        if (c + 1 < p.NT) load_tile(c + 1);
      }
      __syncwarp();
      named_sync(NB_C, kNbC);  // h staged, C_k written
      if (lane == 0) {
        tma_store_4d(&mapH, sH, 0, mt(c) * LT, hh, b);
        tma_store_4d(&mapH, sH + SM::kTile, 64, mt(c) * LT, hh, b);
        if (p.store_states && c + 1 < p.NT) store_state(c + 1);  // C_k = state entering tile c+1
        tma_store_commit();
        tma_store_wait_read<0>();  // the staging tile aliases P: it must be drained before bar_s(c+1) completes
      }
      __syncwarp();
      if (c + 1 < p.NT && elect_one()) issue_s(c + 1);
      __syncwarp();
    }
    if (lane == 0) tma_store_wait_all<0>();
  } else if (warp == kScanWarp) {
    fw_scan_warp<REV, EPI ? D * 2 : 0>(p, ip, fp, mt, fsm + SM::fGates, bar_g,
                                       p.x ? (const uint16_t*)p.x + b * p.x_sb + hh * p.x_sh : nullptr);
  } else {
    // =========================== worker warps ===================================================
    float m_run = p.m0 ? p.m0[bh] : 0.f;
    int cur = 0;
    for (int c = 0; c < p.NT; ++c) {
      const int pb = c & 1;
      const uint32_t par = c & 1;
      const float* gb = fsm + SM::fGates + pb * GateBuf::kFloats;
      float* srs = fsm + SM::fRs + pb * 2 * LT;
      float* sqn = fsm + SM::fQn + pb * 2 * LT;
      float* snp = fsm + SM::fNp + pb * 4 * D;
      const float* sNc = fsm + SM::fN + cur * D;
      float* sNn = fsm + SM::fN + (cur ^ 1) * D;
      const int t0 = mt(c) * LT;
      const int n_valid = min(LT, p.S - t0);

      mbar_wait(&bar_g[pb], (c >> 1) & 1, 2);
      const auto [g, m_next, gbar, b_t, i_t, m_t] = tile_gates(gb, row, m_run, p.sig);
      mbar_wait(&bar_full, par, 3);
      if (c > 0) mbar_wait(&bar_n, (c - 1) & 1, 4);
      {  // partial q . n_{k-1} over this thread's 64 columns
        float qn = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          uint4 q = *reinterpret_cast<const uint4*>(sQ + ch * SM::kTile + swz128(row, 8 * j));
          float2 q0 = unpack2<T>(q.x), q1 = unpack2<T>(q.y), q2 = unpack2<T>(q.z), q3 = unpack2<T>(q.w);
          const float4 n0 = *reinterpret_cast<const float4*>(sNc + ch * 64 + 8 * j);
          const float4 n1 = *reinterpret_cast<const float4*>(sNc + ch * 64 + 8 * j + 4);
          qn += q0.x * n0.x + q0.y * n0.y + q1.x * n0.z + q1.y * n0.w + q2.x * n1.x + q2.y * n1.y + q3.x * n1.z + q3.y * n1.w;
        }
        sqn[ch * LT + row] = qn;
      }
      // ---- P = S . D (causal), row sums; P written swizzled to sP -----------------------------------
      mbar_wait(&bar_s, par, 5);
      tc_fence_after_sync();
      srs[ch * LT + row] = causal_p<REV>(tS + lane_base, gb, b_t, m_t, p.scale, rb, ch, lane,
                                         [&](int u, const float(&v)[32]) { store_row32<T>(sP, row, u * 32, v); });
      fence_proxy_async_smem();
      tc_fence_before_sync();
      named_arrive(NB_B, kNbAB);
      {  // Kbar = abar . K (row, 64 columns in two halves); column sums for n
        const float ab = __expf(g - b_t + i_t - m_next);  // fw.py:102
#pragma unroll 1
        for (int hf = 0; hf < 2; ++hf) {
          float kb[32];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint4 u = *reinterpret_cast<const uint4*>(sK + ch * SM::kTile + swz128(row, hf * 32 + 8 * j));
            float2 a0 = unpack2<T>(u.x), a1 = unpack2<T>(u.y), a2 = unpack2<T>(u.z), a3 = unpack2<T>(u.w);
            kb[8 * j + 0] = a0.x * ab; kb[8 * j + 1] = a0.y * ab; kb[8 * j + 2] = a1.x * ab; kb[8 * j + 3] = a1.y * ab;
            kb[8 * j + 4] = a2.x * ab; kb[8 * j + 5] = a2.y * ab; kb[8 * j + 6] = a3.x * ab; kb[8 * j + 7] = a3.y * ab;
          }
          store_row32<T>(sKb, row, ch * 64 + hf * 32, kb);
          const float cs = warp_colsum32(kb, lane);
          snp[rb * D + ch * 64 + hf * 32 + lane] = cs;
        }
        fence_proxy_async_smem();
        named_arrive(NB_A, kNbAB);
      }
      // ---- epilogue: h (row, 64 columns in two halves) -----------------------------------------------------
      mbar_wait(&bar_h, par, 7);
      tc_fence_after_sync();
      {
        const auto [bq, nmax, inv] = normaliser(
            p, b_t, m_run, m_t, [&](float bq_t) { return bq_t * (sqn[row] + sqn[LT + row]) + srs[row] + srs[LT + row]; });
#pragma unroll 1
        for (int hf = 0; hf < 2; ++hf) {
          uint32_t hi[32], hx[32];
          tmem_ld32_nowait(tHi + lane_base + ch * 64 + hf * 32, hi);
          tmem_ld32_nowait(tHx + lane_base + ch * 64 + hf * 32, hx);
          tmem_ld_wait();
          float o[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] = (__uint_as_float(hi[j]) + bq * __uint_as_float(hx[j])) * inv;  // fw.py:200-212
          store_row32<T>(sH, row, ch * 64 + hf * 32, o);
        }
        if (ch == 0 && row < n_valid) {
          p.n_out[(int64_t)bh * p.S + t0 + row] = nmax;
          p.m_out[(int64_t)bh * p.S + t0 + row] = m_t;
        }
        if (EPI) {  // fused cell output: see tc_fw (this thread: row, columns 64 ch .. 64 ch + 63 = one [128][64] sub-tile)
          uint8_t* sub = sH + ch * SM::kTile;
          const int64_t tok = (int64_t)(t0 + row);
          if (p.h_plain && row < n_valid) {
            uint4* dst = reinterpret_cast<uint4*>((T*)p.h_plain + b * p.h_sb + hh * p.h_sh + tok * p.h_ss + ch * 64);
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[j] = *reinterpret_cast<const uint4*>(sub + swz128(row, 8 * j));
          }
          const void* xrow = p.x ? (const void*)((const uint16_t*)p.x + b * p.x_sb + hh * p.x_sh + tok * p.x_ss + ch * 64) : nullptr;
          // (parameters are indexed by the column inside the head: offset the table instead of the column)
          ln_epilogue_slice<T, 128, 64>(sub, [](int r, int cc) { return swz128(r, cc & 63); }, row, ch * 64, ch, NB_PAIR0 + rb,
                                        fsm + SM::fStat, fsm + SM::fPar, xrow, p.xy_f16 != 0, p.ln_eps, row < n_valid);
        }
      }
      // ---- state update C_k = gbar C_{k-1} + dC (M128 layout: lane == dqk row); n_k -----------------------
      mbar_wait(&bar_dc, par, 6);
      tc_fence_after_sync();
      {
        fw128_update_c<T>(Creg, gbar, tDC + lane_base + ch * 64, sC, row, ch * 64);
        if (tid < D) {  // n_k = gbar n_{k-1} + column sums of Kbar (fw.py:116)
          sNn[tid] = gbar * sNc[tid] + ((snp[tid] + snp[D + tid]) + (snp[2 * D + tid] + snp[3 * D + tid]));
          mbar_arrive(&bar_n);
        }
      }
      fence_proxy_async_smem();
      tc_fence_before_sync();
      named_arrive(NB_C, kNbC);
      m_run = m_next;
      cur ^= 1;
    }
    if (p.c_last) {  // final states (fw.py:302-309)
      float* dst = p.c_last + ((int64_t)bh * D + row) * D + ch * 64;
#pragma unroll
      for (int j = 0; j < 64; ++j) dst[j] = Creg[j];
      if (tid < D) p.n_last[(int64_t)bh * D + tid] = fsm[SM::fN + cur * D + tid];
      if (tid == 0) p.m_last[bh] = m_run;
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == kCtlWarp) tmem_dealloc<512>(tmem);
}

// =============================================================================================
// Forward, wide heads (DHQK, DHHV) = (256, 512): xLSTM-Large's mLSTM layer (qk_dim_factor 0.5, v_dim_factor 1.0) at
// embedding 4096 with 8 heads.  CTA x runs column block vb = x % 8 of v / h / C of (batch, head) x / 8 (the 8 CTAs of a
// head are adjacent, so their Q / K / gate reads meet in L2); n and m do not depend on v, so every block computes them
// and block 0 writes them.  Same algorithm and warp roles as tc_fw_d128, with these differences:
//   * Q and K are resident as four [128][64] swizzled K-blocks (S = Q K^T and Q C have K = 256); v is one 64-wide block.
//   * dC = (abar.K)^T V is computed as K^T (abar.V) -- abar is a per-token factor -- so the scaled operand is the 16 KB
//     V block instead of a 64 KB copy of K: two M128 N64 K128 MMAs (dqk rows 0-127 and 128-255).  dn = K^T abar (the
//     ones-tile MMA of tc_fw with abar in row 0 of the B tile) gives n in fp32 (two M128 N16 MMAs).
//   * P never goes through shared memory (packed into the S columns of TMEM, as tc_fw), and h is written straight from
//     the registers (64 bytes per thread and row), so one Q / K / V stage fits (213 KB); the next tile is pulled into
//     L2 two tiles ahead as in tc_fw_d128.
//   * C: every worker thread owns dqk row 128 ch + row of the 256 x 64 block, 64 fp32 registers (M128 TMEM layout).
// The saved states go out as the four 64 x 64 blocks (qa, vb) of this CTA's column block, in the layout of
// make_states_map_blocks with bd = 64 (rows (8 qa + vb) 64 of a tile), which the 4 x 8 block problems of the backward
// load.  TMEM: S 128 | Hintra 64 | Hinter 64 | dC 2 x 64 | dn 2 x 16 = 416 of 512 columns.
// =============================================================================================
struct FwSmemWide {
  static constexpr int DK = 256, DV = 64, VB = 8;  // DV: the column block of one CTA
  static constexpr int kTile = LT * 128;           // one [128][64] sub-tile
  static constexpr int oQ = 0, oK = 4 * kTile, oV = 8 * kTile;
  static constexpr int oVb = 9 * kTile;            // abar . V
  static constexpr int oC = 10 * kTile;            // bf16 copy of the C block: [256 dqk rows][64 dv cols]
  static constexpr int oA = 12 * kTile;            // abar as row 0 of a K-major [16][128 tokens] B tile (rows 1-15 zero)
  static constexpr int oSmall = oA + 4096;
  // floats: gates[2], srs[2][2][LT], sqn[2][2][LT], sN[2][DK]
  static constexpr int fGates = 0, fRs = 2 * GateBuf::kFloats, fQn = fRs + 4 * LT, fN = fQn + 4 * LT,
                       kSmallFloats = fN + 2 * DK;
  static constexpr int kBytes = oSmall + kSmallFloats * 4 + 1024;
  static constexpr uint32_t kLoadBytes = 9 * kTile;
  static constexpr uint32_t cS = 0, cHi = 128, cHx = 192, cDC = 256, cDN = 384;
  static_assert(kBytes + 1024 <= 228 * 1024, "shared memory");
};

template <typename T, bool REV>
__global__ void __launch_bounds__(kTcThreads, 1)
tc_fw_wide(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
           const __grid_constant__ CUtensorMap mapV, const __grid_constant__ CUtensorMap mapCs, TcFwParams p) {
  using SM = FwSmemWide;
  constexpr int DK = SM::DK, DV = SM::DV, VB = SM::VB;
  constexpr bool kBf16 = std::is_same<T, __nv_bfloat16>::value;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  float* fsm = (float*)(smem + SM::oSmall);
  uint8_t* sQ = smem + SM::oQ;
  uint8_t* sK = smem + SM::oK;
  uint8_t* sV = smem + SM::oV;
  uint8_t* sVb = smem + SM::oVb;
  uint8_t* sC = smem + SM::oC;
  uint8_t* sA = smem + SM::oA;
  __shared__ uint64_t bar_full, bar_s, bar_dc, bar_h, bar_g[2], bar_n;
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int bh = blockIdx.x / VB, vb = blockIdx.x % VB, b = bh / p.NH, hh = bh % p.NH;

  fw128_prologue(warp, bar_full, bar_s, bar_dc, bar_h, bar_g, bar_n, kWorkers, tmem_base_s, mapQ, mapK, mapV, mapCs);
  const int rb = warp & 3, ch = (warp >> 2) & 1;
  const int row = rb * 32 + lane;  // tile row == TMEM lane
  const int drow = ch * 128 + row;  // the dqk row of C (and entry of n) this thread owns
  const uint32_t lane_base = (uint32_t)(rb * 32) << 16;
  float Creg[DV];                  // C[drow][64 vb .. 64 vb + 63], fp32 master copy
#pragma unroll
  for (int j = 0; j < DV; ++j) Creg[j] = 0.f;
  if (warp < kCtlWarp) {
    fw128_load_c0<T>(Creg, p.c0, ((int64_t)bh * DK + drow) * (VB * DV) + vb * DV, sC, drow, 0);
    fsm[SM::fN + tid] = p.n0 ? p.n0[(int64_t)bh * DK + tid] : 0.f;  // kWorkers == DK
    for (int e = tid; e < 4096 / 16; e += kWorkers) reinterpret_cast<uint4*>(sA)[e] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_s;
  const uint32_t tS = tmem + SM::cS, tHi = tmem + SM::cHi, tHx = tmem + SM::cHx, tDC = tmem + SM::cDC, tDN = tmem + SM::cDN;

  const T* ip = (const T*)p.ig + b * p.ig_sb + hh * p.ig_sh;
  const T* fp = (const T*)p.fg + b * p.fg_sb + hh * p.fg_sh;
  auto mt = [&](int c) { return REV ? p.NT - 1 - c : c; };

  if (warp == kCtlWarp) {
    // =========================== control warp ===================================================
    auto load_tile = [&](int c) {
      mbar_expect_tx(&bar_full, SM::kLoadBytes);
#pragma unroll
      for (int kb = 0; kb < 4; ++kb) {
        tma_load_4d(sQ + kb * SM::kTile, &mapQ, &bar_full, kb * 64, mt(c) * LT, hh, b);
        tma_load_4d(sK + kb * SM::kTile, &mapK, &bar_full, kb * 64, mt(c) * LT, hh, b);
      }
      tma_load_4d(sV, &mapV, &bar_full, vb * DV, mt(c) * LT, hh, b);
    };
    auto prefetch_tile = [&](int c) {
#pragma unroll
      for (int kb = 0; kb < 4; ++kb) {
        tma_prefetch_4d(&mapQ, kb * 64, mt(c) * LT, hh, b);
        tma_prefetch_4d(&mapK, kb * 64, mt(c) * LT, hh, b);
      }
      tma_prefetch_4d(&mapV, vb * DV, mt(c) * LT, hh, b);
    };
    constexpr uint32_t id_s = umma_idesc(128, 128, false, false, kBf16);  // Q K^T: A, B K-major
    constexpr uint32_t id_hx = umma_idesc(128, DV, false, true, kBf16);   // Q C: A K-major, B MN-major
    constexpr uint32_t id_h = umma_idesc(128, DV, false, true, kBf16);    // P V: A from TMEM, B MN-major
    constexpr uint32_t id_dc = umma_idesc(128, DV, true, true, kBf16);    // K^T Vbar: A, B MN-major
    constexpr uint32_t id_dn = umma_idesc(128, 16, true, false, kBf16);   // K^T abar: A MN-major, B K-major
    const uint64_t dQ = umma_smem_desc(smem_u32(sQ), 0, 1024), dK = umma_smem_desc(smem_u32(sK), 0, 1024);
    const uint64_t dKm = umma_smem_desc(smem_u32(sK), SM::kTile, 1024);  // K as an MN-major A (dqk 0-127; +2 tiles: 128-255)
    const uint64_t dV = umma_smem_desc(smem_u32(sV), 0, 1024), dVb = umma_smem_desc(smem_u32(sVb), 0, 1024);
    const uint64_t dC = umma_smem_desc(smem_u32(sC), 0, 1024);
    const uint64_t dA = umma_smem_desc(smem_u32(sA), 0, 1024);
    // the four 64 x 64 blocks of the state entering tile c (64 consecutive dqk rows of sC each)
    auto store_state = [&](int c) {
#pragma unroll
      for (int qa = 0; qa < 4; ++qa)
        tma_store_4d(&mapCs, sC + qa * 8192, 0, mt(c) * (4 * VB * 64) + (qa * VB + vb) * 64, hh, b);
    };
    if (lane == 0) {
      if (p.store_states) {
        store_state(0);
        tma_store_commit();
      }
      load_tile(0);
      if (p.NT > 1) prefetch_tile(1);
    }
    __syncwarp();
    for (int c = 0; c < p.NT; ++c) {
      const uint32_t par = c & 1;
      if (lane == 0 && c + 2 < p.NT) prefetch_tile(c + 2);
      __syncwarp();
      if (elect_one()) {
        mbar_wait(&bar_full, par, 1);
        tc_fence_after_sync();
#pragma unroll
        for (int kk = 0; kk < DK / 16; ++kk)  // S = Q K^T
          umma_f16(tS, umma_desc_advance(dQ, (kk / 4) * SM::kTile + (kk % 4) * 32),
                   umma_desc_advance(dK, (kk / 4) * SM::kTile + (kk % 4) * 32), id_s, kk > 0);
        umma_commit(&bar_s);
#pragma unroll
        for (int kk = 0; kk < DK / 16; ++kk)  // Hinter = Q C_{k-1} (sC was written before the previous NB_C)
          umma_f16(tHx, umma_desc_advance(dQ, (kk / 4) * SM::kTile + (kk % 4) * 32), umma_desc_advance(dC, kk * 2048), id_hx,
                   kk > 0);
      }
      __syncwarp();
      named_sync(NB_B, kNbAB);  // P(c) written
      // the store of the state entering tile c has read sC before the workers rewrite it (after bar_dc below)
      if (lane == 0) tma_store_wait_read<0>();
      __syncwarp();
      if (elect_one()) {
        tc_fence_after_sync();
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // Hintra = P V, A = P from TMEM (packed inside the S columns)
          umma_f16_ts(tHi, tS + 32 * (kk / 2) + 8 * (kk % 2), umma_desc_advance(dV, kk * 2048), id_h, kk > 0);
        umma_commit(&bar_h);  // also covers Hinter
      }
      __syncwarp();
      named_sync(NB_A, kNbAB);  // Vbar(c) and abar(c) written
      if (elect_one()) {
#pragma unroll
        for (int hq = 0; hq < 2; ++hq) {
#pragma unroll
          for (int kk = 0; kk < LT / 16; ++kk)  // dC = K^T Vbar, dqk rows 128 hq ..
            umma_f16(tDC + hq * DV, umma_desc_advance(dKm, 2 * hq * SM::kTile + kk * 2048), umma_desc_advance(dVb, kk * 2048),
                     id_dc, kk > 0);
#pragma unroll
          for (int kk = 0; kk < LT / 16; ++kk)  // dn = K^T abar
            umma_f16(tDN + hq * 16, umma_desc_advance(dKm, 2 * hq * SM::kTile + kk * 2048),
                     umma_desc_advance(dA, (kk / 4) * 2048 + (kk % 4) * 32), id_dn, kk > 0);
        }
        umma_commit(&bar_dc);
        mbar_wait(&bar_h, par, 8);  // every MMA of this tile has read Q / K / V: refill the single stage
        mbar_wait(&bar_dc, par, 9);
        if (c + 1 < p.NT) load_tile(c + 1);
      }
      __syncwarp();
      named_sync(NB_C, kNbC);  // h written, C_k written
      if (lane == 0 && p.store_states && c + 1 < p.NT) {
        store_state(c + 1);  // C_k = state entering tile c+1
        tma_store_commit();
      }
      __syncwarp();
    }
    if (lane == 0) tma_store_wait_all<0>();
  } else if (warp == kScanWarp) {
    fw_scan_warp<REV, 0>(p, ip, fp, mt, fsm + SM::fGates, bar_g, nullptr);
  } else {
    // =========================== worker warps ===================================================
    float m_run = p.m0 ? p.m0[bh] : 0.f;
    int cur = 0;
    T* hbase = (T*)p.h_plain + b * p.h_sb + hh * p.h_sh + vb * DV + ch * 32;
    for (int c = 0; c < p.NT; ++c) {
      const int pb = c & 1;
      const uint32_t par = c & 1;
      const float* gb = fsm + SM::fGates + pb * GateBuf::kFloats;
      float* srs = fsm + SM::fRs + pb * 2 * LT;
      float* sqn = fsm + SM::fQn + pb * 2 * LT;
      const float* sNc = fsm + SM::fN + cur * DK;
      float* sNn = fsm + SM::fN + (cur ^ 1) * DK;
      const int t0 = mt(c) * LT;
      const int n_valid = min(LT, p.S - t0);

      mbar_wait(&bar_g[pb], (c >> 1) & 1, 2);
      const auto [g, m_next, gbar, b_t, i_t, m_t] = tile_gates(gb, row, m_run, p.sig);
      mbar_wait(&bar_full, par, 3);
      if (c > 0) mbar_wait(&bar_n, (c - 1) & 1, 4);
      {  // partial q . n_{k-1} over this thread's 128 dqk columns (K-blocks 2 ch, 2 ch + 1)
        float qn = 0.f;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            uint4 q = *reinterpret_cast<const uint4*>(sQ + (2 * ch + hf) * SM::kTile + swz128(row, 8 * j));
            float2 q0 = unpack2<T>(q.x), q1 = unpack2<T>(q.y), q2 = unpack2<T>(q.z), q3 = unpack2<T>(q.w);
            const float* nn = sNc + ch * 128 + hf * 64 + 8 * j;
            const float4 n0 = *reinterpret_cast<const float4*>(nn);
            const float4 n1 = *reinterpret_cast<const float4*>(nn + 4);
            qn += q0.x * n0.x + q0.y * n0.y + q1.x * n0.z + q1.y * n0.w + q2.x * n1.x + q2.y * n1.y + q3.x * n1.z + q3.y * n1.w;
          }
        }
        sqn[ch * LT + row] = qn;
      }
      // ---- P = S . D (causal), row sums, packed into the S columns (as tc_fw) ------------------------
      mbar_wait(&bar_s, par, 5);
      tc_fence_after_sync();
      srs[ch * LT + row] = causal_p<REV>(tS + lane_base, gb, b_t, m_t, p.scale, rb, ch, lane,
                                         [&](int u, const float(&v)[32]) { tmem_st_p<T>(tS + lane_base + u * 32, v); });
      tmem_st_wait();
      tc_fence_before_sync();
      named_arrive(NB_B, kNbAB);
      {  // Vbar = abar . V (row, 32 columns); abar into row 0 of the dn operand
        const float ab = __expf(g - b_t + i_t - m_next);  // fw.py:102 (exp(-inf) = 0 for tail tokens)
        float vb32[32];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 u = *reinterpret_cast<const uint4*>(sV + swz128(row, ch * 32 + 8 * j));
          float2 a0 = unpack2<T>(u.x), a1 = unpack2<T>(u.y), a2 = unpack2<T>(u.z), a3 = unpack2<T>(u.w);
          vb32[8 * j + 0] = a0.x * ab; vb32[8 * j + 1] = a0.y * ab; vb32[8 * j + 2] = a1.x * ab; vb32[8 * j + 3] = a1.y * ab;
          vb32[8 * j + 4] = a2.x * ab; vb32[8 * j + 5] = a2.y * ab; vb32[8 * j + 6] = a3.x * ab; vb32[8 * j + 7] = a3.y * ab;
        }
        store_cols<T, 64>(sVb, row, ch * 32, vb32);
        if (ch == 0) *reinterpret_cast<T*>(sA + (row >> 6) * 2048 + swz128(0, row & 63)) = from_f32<T>(ab);
        fence_proxy_async_smem();
        named_arrive(NB_A, kNbAB);
      }
      // ---- epilogue: h (row, 32 columns) straight to global memory -------------------------------------
      mbar_wait(&bar_h, par, 7);
      tc_fence_after_sync();
      {
        uint32_t hi[32], hx[32];
        tmem_ld32_nowait(tHi + lane_base + ch * 32, hi);
        tmem_ld32_nowait(tHx + lane_base + ch * 32, hx);
        const auto [bq, nmax, inv] = normaliser(
            p, b_t, m_run, m_t, [&](float bq_t) { return bq_t * (sqn[row] + sqn[LT + row]) + srs[row] + srs[LT + row]; });
        tmem_ld_wait();
        if (row < n_valid) {
          uint4* dst = reinterpret_cast<uint4*>(hbase + (int64_t)(t0 + row) * p.h_ss);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float o[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = (__uint_as_float(hi[8 * j + e]) + bq * __uint_as_float(hx[8 * j + e])) * inv;
            uint4 u;
            u.x = pack2<T>(o[0], o[1]);
            u.y = pack2<T>(o[2], o[3]);
            u.z = pack2<T>(o[4], o[5]);
            u.w = pack2<T>(o[6], o[7]);
            dst[j] = u;
          }
          if (ch == 0 && vb == 0) {
            p.n_out[(int64_t)bh * p.S + t0 + row] = nmax;
            p.m_out[(int64_t)bh * p.S + t0 + row] = m_t;
          }
        }
      }
      // ---- state update C_k = gbar C_{k-1} + dC (M128 layout: lane == dqk row within the half); n_k -------
      mbar_wait(&bar_dc, par, 6);
      tc_fence_after_sync();
      {
        uint32_t dn_u;
        tmem_ld1_nowait(tDN + ch * 16 + lane_base, dn_u);
        fw128_update_c<T>(Creg, gbar, tDC + ch * DV + lane_base, sC, drow, 0);  // (its first TMEM load waits for dn_u too)
        sNn[drow] = gbar * sNc[drow] + __uint_as_float(dn_u);  // n_k = gbar n_{k-1} + K^T abar (fw.py:116)
        mbar_arrive(&bar_n);
      }
      fence_proxy_async_smem();
      tc_fence_before_sync();
      named_arrive(NB_C, kNbC);
      m_run = m_next;
      cur ^= 1;
    }
    if (p.c_last) {  // final states (fw.py:302-309)
      float* dst = p.c_last + ((int64_t)bh * DK + drow) * (VB * DV) + vb * DV;
#pragma unroll
      for (int j = 0; j < DV; ++j) dst[j] = Creg[j];
      if (vb == 0) p.n_last[(int64_t)bh * DK + drow] = fsm[SM::fN + cur * DK + drow];  // this thread's own entry
      if (tid == 0 && vb == 0) p.m_last[bh] = m_run;
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == kCtlWarp) tmem_dealloc<512>(tmem);
}

// =============================================================================================
// Backward: one reverse sweep per (batch, head) over 128-token tiles (reference native/bw.py).
// dC lives on chip (fp32 registers + bf16 operand copy); C_{k-1} comes from the forward's
// c_states.  n_out and every max state are constants (bw.py:44-47).  Per tile:
//   S = Q K^T, dSb = dH V^T                      tcgen05 M128 N128 K64 (x2)
//   W = exp(b_t - b_s + i_s - m_t) / (n_t + eps) (s <= t);  Sb' = S.W (scale applied to dV1) ; dS = dSb.W
//   ddC = (wq.Q)^T dH        M64 N64 K128        dQb = dH C_{k-1}^T     M128 N64 K64
//   dQa = dS K               M128 N64 K128       dV1 = Sb'^T dH         M128 N64 K128
//   dV2 = K dC_k             M128 N64 K64        dK1 = dS^T Q           M128 N64 K128
//   dK2 = V dC_k^T           M128 N64 K64
//   dq = scale (dQa + bbar/(n+eps) dQb);  dv = dV1 + abar dV2;  dk = scale dK1 + abar dK2
//   dC_{k-1} = gbar dC_k + ddC;  dI = v.dv;  dF = sigmoid(-f) . suffix-sum(q.dq - k.dk)
// =============================================================================================
struct TcBwParams {
  int B, NH, S, NT;
  float eps, scale;
  const void *ig, *fg;
  int64_t ig_sb, ig_sh, ig_ss, fg_sb, fg_sh, fg_ss;
  const float* m0;
  const float *n_out, *m_out, *dc_last;
  void *di, *df;
  int64_t di_sb, di_sh, di_ss, df_sb, df_sh, df_ss;
  float* dc0;
  int rev;  // 1: the forward ran anti-causally; this sweep then walks the memory tiles in ascending order
  int sig;  // 1: sigmoid input gate (m_out is all zeros, dI picks up sigmoid(-i)); 2: the same without the normaliser
            // (dh is not scaled by 1 / (n + eps), n_out is not read)
  float cap;  // > 0: gate soft cap (see TcFwParams); dI / dF are written w.r.t. the pre-activations
  // head-dim-128 block problems: add into outputs another block problem of the same call has already written
  // (dq / dk / dv through TMA reduce-add, di / df read-modify-write by their one owner thread)
  int acc_qk, acc_v, acc_g;
  // rows of the saved-states matrix per 128-token tile and row offset of this problem's D x D block inside a tile:
  // (D, 0) normally; (256, 64 * block) when a head-dim-128 backward runs as four head-dim-64 block problems
  int cs_rows, cs_off;
#ifdef MLSTM_TC_PROFILE
  long long* prof;
#endif
};

template <int D_>
struct BwSmem {
  static constexpr int D = D_;
  static constexpr int kTile = Lay<D>::kTile;   // one [128][D] tile
  static constexpr int kPTile = LT * 128;       // one [128][64] half of Sb' / dS
  static constexpr int kState = Lay<D>::kState;
  // input ring: kNST stages of [Q | K | V | dH | C_{k-1}].  D = 64 has room for one stage (its tiles are
  // re-filled one by one as the MMA batch releases them); D = 32 prefetches a whole tile ahead.
  static constexpr int kNST = D == 64 ? 1 : 2;
  static constexpr int kStage = 4 * kTile + kState;
  static constexpr int oQ = 0, oK = kTile, oV = 2 * kTile, odH = 3 * kTile, oCs = 4 * kTile;  // inside a stage
  static constexpr int oQt = kNST * kStage;     // wq . Q
  static constexpr int oSb = oQt + kTile;       // Sb' two halves
  static constexpr int odS = oSb + 2 * kPTile;  // dS  two halves
  static constexpr int odQ = odS + 2 * kPTile;  // dq / dv / dk staging (their stores overlap the next tile's W phase)
  static constexpr int odV = odQ + kTile;
  static constexpr int odK = odV + kTile;
  static constexpr int odC = odK + kTile;       // dC_k bf16 operand copy
  static constexpr int oSmall = odC + kState;
  // floats: gates[2], spart[2][6][LT]
  static constexpr int fGates = 0, fPart = 2 * GateBuf::kFloats, kSmallFloats = fPart + 12 * LT;
  static constexpr int kBytes = oSmall + kSmallFloats * 4 + 1024;
  static constexpr uint32_t kLoadBytes = 4 * kTile + kState;
  // TMEM columns.  D = 64: the S / dSb columns are re-used by the dV / dK accumulators.  D = 32: nothing aliases,
  // so S / dSb of the next tile are issued right behind the MMA batch and overlap the epilogues.
  static constexpr bool kAlias = D == 64;
  static constexpr uint32_t cS = 0, cdSb = 128;
  static constexpr uint32_t cdV1 = D == 64 ? 0 : 256, cdV2 = cdV1 + D, cdK1 = D == 64 ? 128 : 320, cdK2 = cdK1 + D,
                            cdQa = D == 64 ? 256 : 384, cdQb = cdQa + D, cddC = D == 64 ? 384 : 448;
};

template <typename T, int D, bool REV, typename TO>
__global__ void __launch_bounds__(kTcThreads, 1)
tc_bw(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
          const __grid_constant__ CUtensorMap mapV, const __grid_constant__ CUtensorMap mapdH,
          const __grid_constant__ CUtensorMap mapCs, const __grid_constant__ CUtensorMap mapdQ,
          const __grid_constant__ CUtensorMap mapdK, const __grid_constant__ CUtensorMap mapdV, TcBwParams p) {
  constexpr bool kBf16 = std::is_same<T, __nv_bfloat16>::value;
  using SM = BwSmem<D>;
  using L = Lay<D>;
  constexpr int CW = L::CW;
  TC_PROF(200, 0);  // kernel entry
  TC_PROF_CTA(0);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQ = smem + SM::oQ;  // stage 0; stage s is SM::kStage bytes further
  uint8_t* sK = smem + SM::oK;
  uint8_t* sV = smem + SM::oV;
  uint8_t* sdH = smem + SM::odH;
  uint8_t* sQt = smem + SM::oQt;
  uint8_t* sSb = smem + SM::oSb;
  uint8_t* sdS = smem + SM::odS;
  uint8_t* sdQ = smem + SM::odQ;
  uint8_t* sdV = smem + SM::odV;
  uint8_t* sdK = smem + SM::odK;
  uint8_t* sCs = smem + SM::oCs;
  uint8_t* sdC = smem + SM::odC;
  float* fsm = (float*)(smem + SM::oSmall);
  __shared__ uint64_t bar_full[SM::kNST], bar_s, bar_q, bar_v, bar_k, bar_d, bar_b, bar_st, bar_g[2];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // provably warp-uniform: role branches stay uniform
  const int bh = blockIdx.x, b = bh / p.NH, hh = bh % p.NH;

  // memory tile of processing tile c (see the forward kernel); the sweep visits c = NT-1 .. 0
  auto mt = [&](int c) { return REV ? p.NT - 1 - c : c; };
  auto load_stage = [&](int s, int c) {  // every input tile of memory tile mt(c) into stage s
    uint8_t* base = smem + s * SM::kStage;
    mbar_expect_tx(&bar_full[s], SM::kLoadBytes);
    tma_load_4d(base + SM::oQ, &mapQ, &bar_full[s], 0, mt(c) * LT, hh, b);
    tma_load_4d(base + SM::oK, &mapK, &bar_full[s], 0, mt(c) * LT, hh, b);
    tma_load_4d(base + SM::oV, &mapV, &bar_full[s], 0, mt(c) * LT, hh, b);
    tma_load_4d(base + SM::odH, &mapdH, &bar_full[s], 0, mt(c) * LT, hh, b);
    tma_load_4d(base + SM::oCs, &mapCs, &bar_full[s], 0, mt(c) * p.cs_rows + p.cs_off, hh, b);
  };
  // cold start: the first input tiles are requested before anything else happens in the CTA (grid-dependency
  // waits: see tc_fw)
  if (tid == kCtlWarp * 32) {
    for (int s = 0; s < SM::kNST; ++s) mbar_init(&bar_full[s], 1);
    fence_mbar_init();
    grid_dep_wait();
    for (int s = 0; s < SM::kNST && s < p.NT; ++s) load_stage(s, p.NT - 1 - s);
  }
  if (tid == 0) {
    mbar_init(&bar_s, 1);
    mbar_init(&bar_b, 1);
    mbar_init(&bar_st, 1);
    mbar_init(&bar_q, 1);
    mbar_init(&bar_v, 1);
    mbar_init(&bar_k, 1);
    mbar_init(&bar_d, 1);
    mbar_init(&bar_g[0], 1);
    mbar_init(&bar_g[1], 1);
    fence_mbar_init();
  }
  if (warp == kCtlWarp) {
    tmem_alloc<512>(&tmem_base_s);
    if (lane == 0) {
      prefetch_tmap(&mapQ); prefetch_tmap(&mapK); prefetch_tmap(&mapV); prefetch_tmap(&mapdH);
      prefetch_tmap(&mapCs); prefetch_tmap(&mapdQ); prefetch_tmap(&mapdK); prefetch_tmap(&mapdV);
    }
  }
  grid_dep_wait();
  grid_dep_launch();
  const int rb = warp & 3, ch = (warp >> 2) & 1;
  const int row = rb * 32 + lane;
  const uint32_t lane_base = (uint32_t)(rb * 32) << 16;
  const int drow = rb * 16 + (lane & 15);
  const bool owns_c = warp < kCtlWarp && lane < 16 && rb * 16 < D;
  float dCreg[CW];
#pragma unroll
  for (int j = 0; j < CW; ++j) dCreg[j] = 0.f;
  if (warp < kCtlWarp) {
    if (p.dc_last && owns_c) {
      const float* src = p.dc_last + ((int64_t)bh * D + drow) * D + ch * CW;
#pragma unroll
      for (int j = 0; j < CW; ++j) dCreg[j] = src[j];
    }
    if (owns_c) store_cols<T, D>(sdC, drow, ch * CW, dCreg);
    fence_proxy_async_smem();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = tmem_base_s;
  const uint32_t tS = tmem + SM::cS, tdSb = tmem + SM::cdSb;
  const uint32_t tdV1 = tmem + SM::cdV1, tdV2 = tmem + SM::cdV2, tdK1 = tmem + SM::cdK1, tdK2 = tmem + SM::cdK2;
  const uint32_t tdQa = tmem + SM::cdQa, tdQb = tmem + SM::cdQb, tddC = tmem + SM::cddC;

  const T* ip = (const T*)p.ig + b * p.ig_sb + hh * p.ig_sh;
  const T* fp = (const T*)p.fg + b * p.fg_sb + hh * p.fg_sh;
  const float* mo = p.m_out + (int64_t)bh * p.S;
  const float* no = p.n_out + (int64_t)bh * p.S;
  if (warp == kCtlWarp) {
    // =========================== control warp ===================================================
    constexpr uint32_t id_s = umma_idesc(128, 128, false, false, kBf16);
    constexpr uint32_t id_c = umma_idesc(64, D, true, true, kBf16);
    constexpr uint32_t id_k_mn = umma_idesc(128, D, false, true, kBf16);   // A K-major, B MN-major
    constexpr uint32_t id_mn_mn = umma_idesc(128, D, true, true, kBf16);   // A MN-major, B MN-major
    constexpr uint32_t id_k_k = umma_idesc(128, D, false, false, kBf16);   // A K-major, B K-major
    // stage-0 descriptors; stage s adds s * kStage (warp-uniform)
    const uint64_t kQ0 = L::desc(smem_u32(sQ), 0), mQ0 = L::desc(smem_u32(sQ), SM::kTile);
    const uint64_t kK0 = L::desc(smem_u32(sK), 0), mK0 = L::desc(smem_u32(sK), SM::kTile);
    const uint64_t kV0 = L::desc(smem_u32(sV), 0);
    const uint64_t kH0 = L::desc(smem_u32(sdH), 0), mH0 = L::desc(smem_u32(sdH), SM::kTile);
    const uint64_t kCs0 = L::desc(smem_u32(sCs), 0);
    const uint64_t mQt = L::desc(smem_u32(sQt), D == 64 ? SM::kTile : 0);  // D = 32: rows 32-63 of the M = 64 MMA re-read the block
    const uint64_t mSb = umma_smem_desc(smem_u32(sSb), SM::kPTile, 1024);
    const uint64_t kdS = umma_smem_desc(smem_u32(sdS), 0, 1024), mdS = umma_smem_desc(smem_u32(sdS), SM::kPTile, 1024);
    const uint64_t kdC = L::desc(smem_u32(sdC), 0), mdC = L::desc(smem_u32(sdC), SM::kState);
    auto issue_s = [&](int it) {  // S = Q K^T, dSb = dH V^T of processing step `it` (its loads are in flight)
      const int s = it % SM::kNST;
      const uint32_t so = (uint32_t)s * SM::kStage;
      const uint64_t kQ = umma_desc_advance(kQ0, so), kK = umma_desc_advance(kK0, so);
      const uint64_t kH = umma_desc_advance(kH0, so), kV = umma_desc_advance(kV0, so);
      mbar_wait(&bar_full[s], (it / SM::kNST) & 1, 11);
      tc_fence_after_sync();
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        umma_f16(tS, umma_desc_advance(kQ, kk * 32), umma_desc_advance(kK, kk * 32), id_s, kk > 0);
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
        umma_f16(tdSb, umma_desc_advance(kH, kk * 32), umma_desc_advance(kV, kk * 32), id_s, kk > 0);
      umma_commit(&bar_s);
    };

    if (elect_one()) issue_s(0);
    __syncwarp();

    for (int it = 0; it < p.NT; ++it) {
      const int c = p.NT - 1 - it, pb = it & 1;
      const uint32_t par = it & 1;
      const int t0 = mt(c) * LT, n_valid = min(LT, p.S - t0);
      const uint32_t so = (uint32_t)(it % SM::kNST) * SM::kStage;
      const uint64_t kQ = umma_desc_advance(kQ0, so), mQ = umma_desc_advance(mQ0, so);
      const uint64_t kK = umma_desc_advance(kK0, so), mK = umma_desc_advance(mK0, so);
      const uint64_t kV = umma_desc_advance(kV0, so), kCs = umma_desc_advance(kCs0, so);
      const uint64_t kH = umma_desc_advance(kH0, so), mH = umma_desc_advance(mH0, so);
      TC_PROF(it, 9);
      if (SM::kNST == 1 && c > 0 && lane == 0) {  // single input stage: pull the next tile into L2 a whole tile ahead,
        const int r = mt(c - 1) * LT;             // so that the re-fills behind the MMA batch are L2 hits
        tma_prefetch_4d(&mapQ, 0, r, hh, b);
        tma_prefetch_4d(&mapK, 0, r, hh, b);
        tma_prefetch_4d(&mapV, 0, r, hh, b);
        tma_prefetch_4d(&mapdH, 0, r, hh, b);
        tma_prefetch_4d(&mapCs, 0, mt(c - 1) * p.cs_rows + p.cs_off, hh, b);
      }
      named_sync(NB_B, kNbAB);  // Sb', dS written
      TC_PROF(it, 10);
      // MMA batch, ordered (a) so that the first epilogue (dk) can start after 12 of the 44 instructions and
      // (b) so that the input tiles die one after the other: each is re-filled with the next tile's rows as soon
      // as its last reader has completed (D = 64, single input stage) instead of idling the CTA on the loads.
      if (elect_one()) {
        tc_fence_after_sync();
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // dK1 = dS^T Q
          umma_f16(tdK1, umma_desc_advance(mdS, kk * 2048), umma_desc_advance(mQ, kk * L::kAdvMN), id_mn_mn, kk > 0);
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk)  // dK2 = V dC_k^T
          umma_f16(tdK2, umma_desc_advance(kV, kk * 32), umma_desc_advance(kdC, kk * 32), id_k_k, kk > 0);
        umma_commit(&bar_k);  // Q, V consumed; dk complete
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // dQa = dS K
          umma_f16(tdQa, umma_desc_advance(kdS, (kk / 4) * SM::kPTile + (kk % 4) * 32), umma_desc_advance(mK, kk * L::kAdvMN),
                   id_k_mn, kk > 0);
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk)  // dQb = dH C_{k-1}^T
          umma_f16(tdQb, umma_desc_advance(kH, kk * 32), umma_desc_advance(kCs, kk * 32), id_k_k, kk > 0);
        umma_commit(&bar_q);  // C_{k-1} consumed; dq complete
#pragma unroll
        for (int kk = 0; kk < D / 16; ++kk)  // dV2 = K dC_k
          umma_f16(tdV2, umma_desc_advance(kK, kk * 32), umma_desc_advance(mdC, kk * L::kAdvMN), id_k_mn, kk > 0);
        umma_commit(&bar_b);  // K consumed
      }
      __syncwarp();
      if (lane == 0) {  // (off the MMA issue path: 128 CTAs store in lockstep, the reads take a while to drain)
        tma_store_wait_read<0>();  // the previous tile's dq / dk / dv stores have left their staging buffers
        mbar_arrive(&bar_st);
      }
      __syncwarp();
      TC_PROF(it, 11);
      named_sync(NB_A, kNbAB);  // Qt written; the workers hold their q / k / v row slices in registers
      TC_PROF(it, 12);
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // ddC = Qt^T dH
          umma_f16(tddC, umma_desc_advance(mQt, kk * L::kAdvMN), umma_desc_advance(mH, kk * L::kAdvMN), id_c, kk > 0);
        umma_commit(&bar_d);
#pragma unroll
        for (int kk = 0; kk < LT / 16; ++kk)  // dV1 = Sb'^T dH
          umma_f16(tdV1, umma_desc_advance(mSb, kk * 2048), umma_desc_advance(mH, kk * L::kAdvMN), id_mn_mn, kk > 0);
        umma_commit(&bar_v);  // dH consumed; dv complete
        if (!SM::kAlias && c > 0) issue_s(it + 1);  // next tile's S / dSb queue up behind the batch
        if (SM::kNST == 1) {
          if (c > 0) {  // re-fill the single stage tile by tile, each as soon as its last reader has completed
            const int r = mt(c - 1) * LT;
            mbar_expect_tx(&bar_full[0], SM::kLoadBytes);
            mbar_wait(&bar_k, par, 21);
            tma_load_4d(sQ, &mapQ, &bar_full[0], 0, r, hh, b);
            tma_load_4d(sV, &mapV, &bar_full[0], 0, r, hh, b);
            mbar_wait(&bar_q, par, 24);
            tma_load_4d(sCs, &mapCs, &bar_full[0], 0, mt(c - 1) * p.cs_rows + p.cs_off, hh, b);
            mbar_wait(&bar_b, par, 22);
            tma_load_4d(sK, &mapK, &bar_full[0], 0, r, hh, b);
            mbar_wait(&bar_v, par, 25);
            tma_load_4d(sdH, &mapdH, &bar_full[0], 0, r, hh, b);
          }
        } else if (c >= SM::kNST) {  // this stage is free once the whole batch has completed
          mbar_wait(&bar_v, par, 25);
          load_stage(it % SM::kNST, c - SM::kNST);
        }
      }
      __syncwarp();
      TC_PROF(it, 13);
      named_sync(NB_C, kNbC);  // dq / dk / dv staged, dC_{k-1} written
      TC_PROF(it, 14);
      if (lane == 0) {
        if (p.acc_qk) {
          tma_reduce_add_4d(&mapdQ, sdQ, 0, t0, hh, b);
          tma_reduce_add_4d(&mapdK, sdK, 0, t0, hh, b);
        } else {
          tma_store_4d(&mapdQ, sdQ, 0, t0, hh, b);
          tma_store_4d(&mapdK, sdK, 0, t0, hh, b);
        }
        if (p.acc_v) tma_reduce_add_4d(&mapdV, sdV, 0, t0, hh, b);
        else tma_store_4d(&mapdV, sdV, 0, t0, hh, b);
        tma_store_commit();
      }
      __syncwarp();
      if (SM::kAlias && c > 0 && elect_one()) issue_s(it + 1);  // S / dSb of the next tile (their TMEM columns were read by this epilogue)
      __syncwarp();
    }
    if (lane == 0) tma_store_wait_all<0>();
  } else if (warp == kScanWarp) {
    // =========================== scan warp: tile vectors two tiles ahead + dI / dF ==================
    // raw per-tile vectors (gate inputs, saved m / n) are loaded one tile before they are scanned
    struct TileRaw {
      GateRaw<T> g;
      float4 mt, nt;
      float m_prev, m_next;
    };
    auto raw_of = [&](int c) {
      TileRaw r;
      const int t0 = mt(c) * LT, n_valid = min(LT, p.S - t0);
      r.g = load_gate_raw<T>(ip + (int64_t)t0 * p.ig_ss, p.ig_ss, fp + (int64_t)t0 * p.fg_ss, p.fg_ss, n_valid);
      if (lane * 4 < n_valid) {  // n_valid is a multiple of 4 (tensor_supported)
        r.mt = *reinterpret_cast<const float4*>(mo + t0 + lane * 4);
        r.nt = p.sig == 2 ? make_float4(1.f, 1.f, 1.f, 1.f) : *reinterpret_cast<const float4*>(no + t0 + lane * 4);
      } else {
        r.mt = make_float4(0.f, 0.f, 0.f, 0.f);
        r.nt = make_float4(1.f, 1.f, 1.f, 1.f);
      }
      // m of the state entering the tile = m_out of the previously processed token; m of the state leaving it
      // = m_out of the tile's last processed token (its first memory row in the anti-causal direction)
      if (!REV) {
        r.m_prev = c > 0 ? mo[t0 - 1] : (p.m0 ? p.m0[bh] : 0.f);
        r.m_next = mo[t0 + n_valid - 1];
      } else {
        r.m_prev = c > 0 ? mo[t0 + LT] : (p.m0 ? p.m0[bh] : 0.f);
        r.m_next = mo[t0];
      }
      return r;
    };
    auto publish = [&](float* gb, const TileRaw& r) {
      gate_scan_regs(gb, r.g, REV, p.sig != 0, p.cap);
      reinterpret_cast<float4*>(gb + GateBuf::oMt)[lane] = r.mt;
      reinterpret_cast<float4*>(gb + GateBuf::oNt)[lane] = r.nt;
      if (lane == 0) {
        gb[GateBuf::oScal + 2] = r.m_prev;
        gb[GateBuf::oScal + 3] = r.m_next;
      }
    };

    TileRaw raw = raw_of(p.NT - 1);
    float carry = 0.f;  // running suffix sum of (q.dq - k.dk)
    // n = processing index of the tile whose vectors are published; the dI / dF scan lags two tiles
    for (int n = 0; n < p.NT + 2; ++n) {
      if (n >= 2) {
      const int it = n - 2;
      const int c = p.NT - 1 - it, pb = it & 1;
      const int t0 = mt(c) * LT, n_valid = min(LT, p.S - t0);
      named_sync(NB_C, kNbC);  // row dots of tile `it` are in shared memory; its buffers can be reused afterwards
      // ---- gate gradients: reverse (suffix) scan over the tile, carried across tiles -------------
      {
        const float* sp = fsm + SM::fPart + pb * 6 * LT;
        const float* gb = fsm + SM::fGates + pb * GateBuf::kFloats;
        float acc[4], di[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int t = lane * 4 + e;
          acc[e] = (sp[0 * LT + t] + sp[1 * LT + t]) - (sp[2 * LT + t] + sp[3 * LT + t]);  // bw.py:321
          di[e] = sp[4 * LT + t] + sp[5 * LT + t];                                         // bw.py:326
        }
        // sum over all tokens processed AFTER t: a suffix sum over memory rows, or a prefix sum when the
        // forward ran anti-causally (this sweep then visits the memory tiles in ascending order)
        float incl, own;
        if (!REV) {
          acc[2] += acc[3];
          acc[1] += acc[2];
          acc[0] += acc[1];
          incl = own = acc[0];
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            float u = __shfl_down_sync(0xffffffffu, incl, o);
            if (lane + o < 32) incl += u;
          }
        } else {
          acc[1] += acc[0];
          acc[2] += acc[1];
          acc[3] += acc[2];
          incl = own = acc[3];
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            float u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
          }
        }
        const float excl = incl - own + carry;
        TO* dip = (TO*)p.di + b * p.di_sb + hh * p.di_sh;
        TO* dfp = (TO*)p.df + b * p.df_sb + hh * p.df_sh;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int t = lane * 4 + e;
          if (t < n_valid) {
            const float dsig = p.sig ? 1.f - __expf(gb[GateBuf::oI + t]) : 1.f;  // sigmoid(-i) = 1 - exp(logsigmoid(i))
            float gi = di[e] * dsig * gb[GateBuf::oDi + t];
            float gf = (acc[e] + excl) * sigmoid_neg_f32(gb[GateBuf::oF + t]) * gb[GateBuf::oDf + t];  // bw.py:322-323
            TO* pi = dip + (int64_t)(t0 + t) * p.di_ss;
            TO* pf = dfp + (int64_t)(t0 + t) * p.df_ss;
            if (p.acc_g) {  // (the block problems of one call run one after the other on the stream)
              gi += to_f32<TO>(*pi);
              gf += to_f32<TO>(*pf);
            }
            *pi = from_f32<TO>(gi);
            *pf = from_f32<TO>(gf);
          }
        }
        carry += __shfl_sync(0xffffffffu, incl, REV ? 31 : 0);
      }
      __syncwarp();
      }
      if (n < p.NT) {
        publish(fsm + SM::fGates + (n & 1) * GateBuf::kFloats, raw);
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_g[n & 1]);
        if (n + 1 < p.NT) raw = raw_of(p.NT - 2 - n);
      }
    }
  } else {
    // =========================== worker warps ===================================================
    for (int it = 0; it < p.NT; ++it) {
      const int pb = it & 1;
      const uint32_t par = it & 1;
      const float* gb = fsm + SM::fGates + pb * GateBuf::kFloats;
      float* spart = fsm + SM::fPart + pb * 6 * LT;
      const int n_valid = min(LT, p.S - mt(p.NT - 1 - it) * LT);
      const bool valid = row < n_valid;
      const uint32_t so = (uint32_t)(it % SM::kNST) * SM::kStage;  // input stage of this tile

      TC_PROF(it, 0);
      mbar_wait(&bar_g[pb], (it >> 1) & 1, 12);
      const float g = gb[GateBuf::oScal], m_prev = gb[GateBuf::oScal + 2], m_next = gb[GateBuf::oScal + 3];
      const float b_t = gb[GateBuf::oB + row], i_t = gb[GateBuf::oI + row];
      const float m_t = gb[GateBuf::oMt + row], n_t = gb[GateBuf::oNt + row];
      const float rinv = !valid ? 0.f : p.sig == 2 ? 1.f : 1.f / (n_t + p.eps);  // bw.py:135 (siging = 2: no normaliser)
      const float bbar = valid ? __expf(b_t + m_prev - m_t) : 0.f;  // bw.py:186
      const float abar = __expf(g - b_t + i_t - m_next);            // bw.py:187 (0 for tail tokens)
      const float gbar = __expf(g + m_prev - m_next);               // bw.py:76
      TC_PROF(it, 1);
      // ---- Qt = wq . Q, written while the S / dSb MMAs of this tile run (ddC of the previous tile, the last
      // reader of sQt, completed before the previous dC update); q row slice kept for the gate gradients
      mbar_wait(&bar_full[it % SM::kNST], (it / SM::kNST) & 1, 13);
      uint32_t qs[CW / 2];
      {
        const float wq = p.scale * bbar * rinv;  // bw.py:83-90
#pragma unroll
        for (int j = 0; j < CW / 8; ++j) {
          const uint32_t off = L::swz(row, ch * CW + 8 * j);
          uint4 u = *reinterpret_cast<const uint4*>(sQ + so + off);
          qs[4 * j] = u.x; qs[4 * j + 1] = u.y; qs[4 * j + 2] = u.z; qs[4 * j + 3] = u.w;
          float2 a0 = unpack2<T>(u.x), a1 = unpack2<T>(u.y), a2 = unpack2<T>(u.z), a3 = unpack2<T>(u.w);
          u.x = pack2<T>(a0.x * wq, a0.y * wq);
          u.y = pack2<T>(a1.x * wq, a1.y * wq);
          u.z = pack2<T>(a2.x * wq, a2.y * wq);
          u.w = pack2<T>(a3.x * wq, a3.y * wq);
          *reinterpret_cast<uint4*>(sQt + off) = u;
        }
      }
      // ---- W = D / (n + eps); Sb' = S.W, dS = dSb.W ------------------------------------------------
      mbar_wait(&bar_s, par, 14);
      tc_fence_after_sync();
      TC_PROF(it, 2);
      {
        // the 1/(n+eps) and scale factors ride in the exponent: W = 2^(x_t + y_s)
        const float x_t = valid ? (b_t - m_t) * kLog2e + log2f(rinv) : -INFINITY;
        const float* sy = gb + GateBuf::oY;
        const float* scf = gb + GateBuf::oCf;
#pragma unroll 1
        for (int u = ch; u < 4; u += 2) {  // this thread's two 32-column units (warp-uniform branches)
          float v[32], w[32];
          if (REV ? u >= rb : u <= rb) {
            uint32_t rv[32], rw[32];
            tmem_ld32_nowait(tS + lane_base + u * 32, rv);
            tmem_ld32_nowait(tdSb + lane_base + u * 32, rw);
            tmem_ld_wait();
            if (u != rb) {  // fully unmasked 32x32 block: rank-1 decay, one exp per row
              const float r_t = ex2_approx(x_t + gb[GateBuf::oScal + 4 + u]);
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4) {
                const float4 cf = *reinterpret_cast<const float4*>(scf + u * 32 + 4 * j4);
                const float cc[4] = {cf.x, cf.y, cf.z, cf.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const int j = 4 * j4 + e;
                  const float wg = cc[e] * r_t;
                  v[j] = __uint_as_float(rv[j]) * wg;  // the scale factor of Sb' is applied in the dv epilogue
                  w[j] = __uint_as_float(rw[j]) * wg;
                }
              }
            } else {  // diagonal block: causal mask, one exp per entry
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4) {
                const float4 y = *reinterpret_cast<const float4*>(sy + u * 32 + 4 * j4);
                const float yy[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const int j = 4 * j4 + e;
                  float wg = ex2_approx(x_t + yy[e]);
                  wg = (REV ? j >= lane : j <= lane) ? wg : 0.f;
                  v[j] = __uint_as_float(rv[j]) * wg;
                  w[j] = __uint_as_float(rw[j]) * wg;
                }
              }
            }
          } else {
            if (it > 0) continue;  // blocks above the diagonal stay zero: written once, by the first tile
#pragma unroll
            for (int j = 0; j < 32; ++j) { v[j] = 0.f; w[j] = 0.f; }
          }
          store_row32<T>(sSb, row, u * 32, v);
          store_row32<T>(sdS, row, u * 32, w);
        }
      }
      fence_proxy_async_smem();
      tc_fence_before_sync();
      named_arrive(NB_B, kNbAB);
      TC_PROF(it, 3);
      // ---- this thread's k / v row slices for the gate gradients (the inputs may be re-filled afterwards) --
      uint32_t ks[CW / 2], vs[CW / 2];
#pragma unroll
      for (int j = 0; j < CW / 8; ++j) {
        const uint32_t off = L::swz(row, ch * CW + 8 * j);
        uint4 uk = *reinterpret_cast<const uint4*>(sK + so + off);
        ks[4 * j] = uk.x; ks[4 * j + 1] = uk.y; ks[4 * j + 2] = uk.z; ks[4 * j + 3] = uk.w;
        uint4 uv = *reinterpret_cast<const uint4*>(sV + so + off);
        vs[4 * j] = uv.x; vs[4 * j + 1] = uv.y; vs[4 * j + 2] = uv.z; vs[4 * j + 3] = uv.w;
      }
      fence_proxy_async_smem();
      named_arrive(NB_A, kNbAB);
      TC_PROF(it, 4);
      // ---- epilogues, pipelined with the MMA batch through three commits ------------------------------
      {
        uint32_t ra[CW], rq[CW];
        float o[CW];
        float dot;
        // dk
        mbar_wait(&bar_k, par, 18);
        tc_fence_after_sync();
        TC_PROF(it, 5);
        tmem_ld_nowait(tdK1 + lane_base + ch * CW, ra);
        tmem_ld_nowait(tdK2 + lane_base + ch * CW, rq);
        tmem_ld_wait();
        dot = 0.f;
#pragma unroll
        for (int j = 0; j < CW / 2; ++j) {
          o[2 * j] = p.scale * __uint_as_float(ra[2 * j]) + abar * __uint_as_float(rq[2 * j]);  // bw.py:170,192
          o[2 * j + 1] = p.scale * __uint_as_float(ra[2 * j + 1]) + abar * __uint_as_float(rq[2 * j + 1]);
          float2 kv = unpack2<T>(ks[j]);
          dot += kv.x * o[2 * j] + kv.y * o[2 * j + 1];
        }
        mbar_wait(&bar_st, par, 19);  // staging buffers free (the previous tile's stores have read them)
        store_cols<TO, D>(sdK, row, ch * CW, o);
        spart[(1 * 2 + ch) * LT + row] = dot;
        // dq
        mbar_wait(&bar_q, par, 16);
        tc_fence_after_sync();
        TC_PROF(it, 6);
        tmem_ld_nowait(tdQa + lane_base + ch * CW, ra);
        tmem_ld_nowait(tdQb + lane_base + ch * CW, rq);
        tmem_ld_wait();
        const float wb = bbar * rinv;
        dot = 0.f;
#pragma unroll
        for (int j = 0; j < CW / 2; ++j) {
          o[2 * j] = p.scale * (__uint_as_float(ra[2 * j]) + wb * __uint_as_float(rq[2 * j]));  // bw.py:169,193
          o[2 * j + 1] = p.scale * (__uint_as_float(ra[2 * j + 1]) + wb * __uint_as_float(rq[2 * j + 1]));
          float2 qv = unpack2<T>(qs[j]);
          dot += qv.x * o[2 * j] + qv.y * o[2 * j + 1];
        }
        store_cols<TO, D>(sdQ, row, ch * CW, o);
        spart[(0 * 2 + ch) * LT + row] = dot;
      }
      // ---- dC_{k-1} = gbar dC_k + ddC ----------------------------------------------------------------
      mbar_wait(&bar_d, par, 15);
      tc_fence_after_sync();
      TC_PROF(it, 7);
      {
        float v[CW];
        tmem_ld(tddC + lane_base + ch * CW, v);
        if (owns_c) {
#pragma unroll
          for (int j = 0; j < CW; ++j) dCreg[j] = gbar * dCreg[j] + v[j];  // bw.py:93-95
          store_cols<T, D>(sdC, drow, ch * CW, dCreg);                     // dV2 / dK2 have completed (bar_k)
        }
      }
      // ---- dv last: dV1 = Sb'^T dH is the final MMA group of the batch ---------------------------------
      {
        uint32_t ra[CW], rq[CW];
        float o[CW];
        float dot;
        // dv
        mbar_wait(&bar_v, par, 17);
        tc_fence_after_sync();
        tmem_ld_nowait(tdV1 + lane_base + ch * CW, ra);
        tmem_ld_nowait(tdV2 + lane_base + ch * CW, rq);
        tmem_ld_wait();
        dot = 0.f;
#pragma unroll
        for (int j = 0; j < CW / 2; ++j) {
          o[2 * j] = p.scale * __uint_as_float(ra[2 * j]) + abar * __uint_as_float(rq[2 * j]);  // bw.py:164,190
          o[2 * j + 1] = p.scale * __uint_as_float(ra[2 * j + 1]) + abar * __uint_as_float(rq[2 * j + 1]);
          float2 vv = unpack2<T>(vs[j]);
          dot += vv.x * o[2 * j] + vv.y * o[2 * j + 1];
        }
        store_cols<TO, D>(sdV, row, ch * CW, o);
        spart[(2 * 2 + ch) * LT + row] = dot;
      }
      fence_proxy_async_smem();
      tc_fence_before_sync();
      named_arrive(NB_C, kNbC);
      TC_PROF(it, 8);
    }
    if (p.dc0 && owns_c) {  // dC_initial = dC_0 (bw.py:329-331)
      float* dst = p.dc0 + ((int64_t)bh * D + drow) * D + ch * CW;
#pragma unroll
      for (int j = 0; j < CW; ++j) dst[j] = dCreg[j];
    }
  }
  TC_PROF(200, 1);  // this role is done
  tc_fence_before_sync();
  __syncthreads();
  TC_PROF(200, 2);
  TC_PROF_CTA(1);
  if (warp == kCtlWarp) tmem_dealloc<512>(tmem);
}

#ifdef MLSTM_TC_PROFILE
// Phase-clock buffer of the PROFILE build only (lib/libmlstm_b200_prof.so, tools/phase_clocks.py); the product
// library carries no process-global mutable state: tensor_set_clock_buffer is a no-op there.
std::atomic<long long*> g_prof{nullptr};
#define TC_SET_PROF(p, off) (p).prof = g_prof.load() ? g_prof.load() + (off) : nullptr
#else
#define TC_SET_PROF(p, off)
#endif

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device) instead of on every launch
// (a runtime call of a few microseconds on the host path of a launch-bound training step)
template <typename K>
cudaError_t ensure_smem(K kern, int bytes) {
  static std::mutex mu;
  static std::set<std::pair<const void*, int>> done;
  int dev = 0;
  cudaGetDevice(&dev);
  const std::pair<const void*, int> key(reinterpret_cast<const void*>(kern), dev);
  {
    std::lock_guard<std::mutex> g(mu);
    if (done.count(key)) return cudaSuccess;
  }
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) {
    std::lock_guard<std::mutex> g(mu);
    done.insert(key);
  }
  return e;
}

// Programmatic dependent launch for the two main kernels (tc_fw, tc_bw): the next kernel's CTAs may become resident
// while this one drains; they block in griddepcontrol.wait before touching memory.  MLSTM_B200_PDL=0 disables it.
int pdl_mode() {  // 0 off, 1 forward and backward, 2 forward only
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MLSTM_B200_PDL");
    v = e ? (e[0] - '0') : 2;
    if (v < 0 || v > 2) v = 2;
  }
  return v;
}
// cudaLaunchKernelEx with programmatic stream serialisation (use_pdl) and, with pair, the two column blocks of a head
// (adjacent CTAs) as one {2, 1, 1} cluster: co-scheduled, and each can reach the other's shared memory.
template <typename... KArgs, typename... Args>
cudaError_t launch_ex(bool use_pdl, bool pair, void (*kern)(KArgs...), int grid, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid), cfg.blockDim = dim3(kTcThreads), cfg.dynamicSmemBytes = smem, cfg.stream = st;
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (pair) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = 2, attr[n].val.clusterDim.y = 1, attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (use_pdl) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr, cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// The call's 16-bit element type and square head dim 32 / 64 as types: f(T{}), g(std::integral_constant<int, D>{})
template <typename F>
int with_dtype(int dtype, F f) {
  return dtype == MLSTM_B200_BF16 ? f(__nv_bfloat16{}) : f(__half{});
}
template <typename F>
int with_d32_64(int D, F f) {
  return D == 32 ? f(std::integral_constant<int, 32>{}) : f(std::integral_constant<int, 64>{});
}
// The instantiation of a forward kernel template for the call's (epi, rev): pick(std::bool_constant<EPI>,
// std::bool_constant<REV>) returns it.  The fused cell-output epilogue is a template parameter: the plain kernel carries
// none of its code (the worker loop is several instruction-cache lines shorter: 33.7 vs 34.3 us at config 2).
template <typename Pick>
auto fw_kernel(bool epi, bool rev, Pick pick) {
  using F = std::false_type;
  using TT = std::true_type;
  return epi ? (rev ? pick(TT{}, TT{}) : pick(TT{}, F{})) : (rev ? pick(F{}, TT{}) : pick(F{}, F{}));
}

// One forward launch of ctas_per_head CTAs per (batch, head); maps: the kernel's tensor maps, in its parameter order.
template <typename K, typename... Maps>
int launch_fw(K kern, const TcFwParams& p, int ctas_per_head, int smem, bool pair, bool use_pdl, cudaStream_t st,
              const Maps&... maps) {
  MLSTM_CUDA_CHECK(ensure_smem(kern, smem));
  MLSTM_CUDA_CHECK(launch_ex(use_pdl, pair, kern, ctas_per_head * p.B * p.NH, smem, st, maps..., p));
  count_launch();
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

template <typename T, int D, typename TO = T>
int launch_bw(const TcBwParams& p, const CUtensorMap& mq, const CUtensorMap& mk, const CUtensorMap& mv,
              const CUtensorMap& mdh, const CUtensorMap& mcs, const CUtensorMap& mdq, const CUtensorMap& mdk,
              const CUtensorMap& mdv, cudaStream_t st) {
  using SM = BwSmem<D>;
  auto kern = p.rev ? tc_bw<T, D, true, TO> : tc_bw<T, D, false, TO>;
  MLSTM_CUDA_CHECK(ensure_smem(kern, SM::kBytes));
  MLSTM_CUDA_CHECK(launch_ex(pdl_mode() == 1, false, kern, p.B * p.NH, SM::kBytes, st, mq, mk, mv, mdh, mcs, mdq, mdk, mdv, p));
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

bool tma_ok(const mlstm_b200_tensor& t) {
  return ((uintptr_t)t.ptr & 15) == 0 && t.stride[3] == 1 && (t.stride[0] % 8) == 0 && (t.stride[1] % 8) == 0 &&
         (t.stride[2] % 8) == 0;
}

// [128 tokens][min(D, 64)] boxes: D = 32 -> 64-byte rows / SWIZZLE_64B, otherwise 128-byte rows / SWIZZLE_128B.
// `box` < D: D-wide rows read or written in box-wide column blocks (v / h of the rectangular and wide forwards).
int make_map(CUtensorMap* m, const mlstm_b200_tensor& t, const mlstm_b200_shape& s, int D, int box = 0) {
  return sm100_host::make_map_bhsd(m, t.ptr, s.dtype == MLSTM_B200_BF16, s.B, s.NH, s.S, D, t.stride[0], t.stride[1],
                                   t.stride[2], LT, box ? box : D == 32 ? 32 : 64);
}

// c_states: the state entering every tile stored as bd x bd blocks, (B, NH, NT * rows, bd) 16-bit with `rows` = nq nv bd
// rows per tile and block (a, b) of a tile at rows (a nv + b) bd (tc_fw_d128::store_state, tc_fw_rect, tc_fw_wide).  A
// square head is block 0 of 1: one [D][D] box per tile.
int make_states_map_blocks(CUtensorMap* m, const void* ptr, const mlstm_b200_shape& s, int rows, int bd) {
  const int NT = (s.S + LT - 1) / LT;
  return sm100_host::make_map_bhsd(m, ptr, s.dtype == MLSTM_B200_BF16, s.B, s.NH, NT * rows, bd, (int64_t)s.NH * NT * rows * bd,
                                   (int64_t)NT * rows * bd, bd, bd, bd);
}

enum class TcFw { none, square, d128, rect, wide };  // the forward kernel families (none: not on the tensor-core route)

// How the tensor-core route cuts a head geometry: a (DHQK, DHHV) head is an nq x nv grid of bd x bd blocks.  The forward
// reads and writes v / h in bd-wide column boxes and stores each tile's state as those blocks (make_states_map_blocks);
// the backward runs one tc_bw<bd> problem per block (bw_by_blocks), or one native problem when the grid is 1 x 1.
struct TcGeometry {
  TcFw fw;
  int bd, nq, nv;
  int ctas;         // forward CTAs per (batch, head)
  bool epilogue;    // the fused cell-output epilogue exists ...
  bool cluster;     // ... and exchanges LayerNorm statistics between the two CTAs of a head: a {2, 1, 1} cluster
  bool gate_parts;  // the backward sums the block problems' dI / dF in fp32 (k_sum_gate_partials)
};

// The one place that knows which (DHQK, DHHV) the tensor-core kernels cover and how each is cut.
TcGeometry tc_geometry(const mlstm_b200_shape& s) {
  // Tiles are 128 tokens whatever chunk_size is (h and the states do not depend on it: the stabiliser equals the
  // step-recurrent one), and ragged last tiles are handled in-kernel (TMA zero-fill, gates masked at scan time),
  // so any S that keeps the fp32 n_out / m_out rows 16-byte aligned is covered; S % chunk_size == 0 is enforced
  // at the C-ABI like the reference does (native/fw.py:252-254).
  if ((s.dtype != MLSTM_B200_BF16 && s.dtype != MLSTM_B200_F16) || s.S % 4 != 0) return {TcFw::none};
  const int dk = s.DHQK, dv = s.DHHV;
  const bool d32_64 = dk == 32 || dk == 64;
  //                                       fw          bd  nq nv  ctas            epilogue cluster gate_parts
  if (d32_64 && dv == dk)       return {TcFw::square, dk, 1, 1, 1,              true,    false,  false};
  // a 128-wide tile set does not fit the backward's shared memory with 128-token tiles: 2 x 2 blocks of 64
  if (dk == 128 && dv == 128)   return {TcFw::d128,   64, 2, 2, 1,              true,    false,  false};
  if (d32_64 && dv == 2 * dk)   return {TcFw::rect,   dk, 1, 2, 2,              true,    true,   false};
  // xLSTM-Large; the in-kernel accumulation of dI / dF would round their running sum to 16 bits 31 times
  if (dk == 256 && dv == 512)   return {TcFw::wide,   64, 4, 8, FwSmemWide::VB, false,   false,  true};
  return {TcFw::none};
}

// Gate, scale and direction fields that TcFwParams and TcBwParams share
template <typename P>
void set_gate_params(P& p, const mlstm_b200_shape& s, const mlstm_b200_tensor& i, const mlstm_b200_tensor& f) {
  p.B = s.B; p.NH = s.NH; p.S = s.S; p.NT = (s.S + LT - 1) / LT;
  p.eps = s.eps;
  p.scale = s.qk_scale > 0.f ? s.qk_scale : 1.f / sqrtf((float)s.DHQK);
  p.ig = i.ptr; p.ig_sb = i.stride[0]; p.ig_sh = i.stride[1]; p.ig_ss = i.stride[2];
  p.fg = f.ptr; p.fg_sb = f.stride[0]; p.fg_sh = f.stride[1]; p.fg_ss = f.stride[2];
  p.rev = s.reverse ? 1 : 0;
  p.sig = s.siging;  // 0, 1 or 2 (checked at the C-ABI)
  p.cap = s.gate_soft_cap;
}

// Forward parameters of a call that stores the state entering every tile into c_states (NULL: no states)
TcFwParams fw_params(const mlstm_b200_fw_args& a, const void* c_states) {
  TcFwParams p{};
  set_gate_params(p, a.shape, a.i, a.f);
  p.c0 = a.c_initial; p.n0 = a.n_initial; p.m0 = a.m_initial;
  p.n_out = a.n_out; p.m_out = a.m_out;
  p.c_last = a.c_last; p.n_last = a.n_last; p.m_last = a.m_last;
  p.store_states = c_states != nullptr;
  // h stored from the registers: always by tc_fw_wide, by the other kernels only with the fused epilogue
  p.h_plain = a.h.ptr; p.h_sb = a.h.stride[0]; p.h_sh = a.h.stride[1]; p.h_ss = a.h.stride[2];
  if (const mlstm_b200_fw_epilogue* ep = a.epilogue) {
    p.epi = 1;
    p.xy_f16 = ep->xy_dtype == MLSTM_B200_F16;
    p.ln_eps = ep->eps;
    p.ln_w = ep->weight; p.ln_b = ep->bias; p.ln_skip = ep->skip;
    p.x = ep->x.ptr; p.x_sb = ep->x.stride[0]; p.x_sh = ep->x.stride[1]; p.x_ss = ep->x.stride[2];
  }
  TC_SET_PROF(p, 0);
  return p;
}

template <typename T, int D>
auto fw_rect_kernel(bool epi, bool rev) {
  return fw_kernel(epi, rev, [](auto e, auto r) { return tc_fw_rect<T, D, decltype(r)::value, decltype(e)::value>; });
}

int run_fw(const mlstm_b200_fw_args& a, void* c_states, cudaStream_t st) {
  const mlstm_b200_shape& s = a.shape;
  const TcGeometry g = tc_geometry(s);
  const mlstm_b200_fw_epilogue* ep = a.epilogue;
  if (ep && !g.epilogue) {
    set_error("the fused cell-output epilogue does not cover (DHQK, DHHV) = (%d, %d)", s.DHQK, s.DHHV);
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (!tensor_views_ok(a)) {
    set_error("tensor path needs 16-byte aligned q/k/v/h with strides that are multiples of 8 elements");
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (ep) {
    if (ep->xy_dtype != MLSTM_B200_BF16 && ep->xy_dtype != MLSTM_B200_F16) {
      set_error("fused epilogue: y / x must be bf16 or fp16");
      return MLSTM_B200_EUNSUPPORTED;
    }
    if ((ep->x.ptr && !tma_ok(ep->x)) || (a.h.ptr && !tma_ok(a.h))) {
      set_error("fused epilogue: x and h need 16-byte aligned rows (unit innermost stride, strides multiples of 8 elements)");
      return MLSTM_B200_EUNSUPPORTED;
    }
  }
  // with the fused epilogue the h map describes y (the un-normalised h, if wanted, is stored from registers); tc_fw_wide
  // stores h from the registers and takes no h map
  const mlstm_b200_tensor& out = ep ? ep->y : a.h;
  mlstm_b200_shape so = s;  // the y map carries y's element type
  if (ep) so.dtype = ep->xy_dtype;
  CUtensorMap mq, mk, mv, mh, mcs;
  int r = make_map(&mq, a.q, s, s.DHQK) | make_map(&mk, a.k, s, s.DHQK) | make_map(&mv, a.v, s, s.DHHV, g.bd) |
          make_map(&mh, out, so, s.DHHV, g.bd);
  // without a c_states buffer the map is never used by the kernel; a copy of the h map keeps it valid
  if (c_states)
    r |= make_states_map_blocks(&mcs, c_states, s, g.nq * g.nv * g.bd, g.bd);
  else
    mcs = mh;
  if (r) {
    set_error("cuTensorMapEncodeTiled failed (%d)", r);
    return MLSTM_B200_ENODEVICE;
  }
  const TcFwParams p = fw_params(a, c_states);
  const bool epi = p.epi != 0, rev = p.rev != 0, pdl = pdl_mode() != 0;
  return with_dtype(s.dtype, [&](auto t) {
    using T = decltype(t);
    switch (g.fw) {
      case TcFw::wide: {
        auto kern = fw_kernel(false, rev, [](auto, auto r) { return tc_fw_wide<T, decltype(r)::value>; });
        return launch_fw(kern, p, g.ctas, FwSmemWide::kBytes, false, false, st, mq, mk, mv, mcs);
      }
      case TcFw::d128: {
        auto kern = fw_kernel(epi, rev, [](auto e, auto r) { return tc_fw_d128<T, decltype(r)::value, decltype(e)::value>; });
        return launch_fw(kern, p, g.ctas, FwSmem128::kBytes, false, false, st, mq, mk, mv, mh, mcs);
      }
      case TcFw::rect:
        return with_d32_64(g.bd, [&](auto d) {
          constexpr int D = decltype(d)::value;
          const bool pair = epi && g.cluster;
          return launch_fw(fw_rect_kernel<T, D>(epi, rev), p, g.ctas, pair ? FwSmem<D>::kBytesPair : FwSmem<D>::kBytes, pair,
                           pdl, st, mq, mk, mv, mh, mcs);
        });
      default:  // TcFw::square
        return with_d32_64(g.bd, [&](auto d) {
          constexpr int D = decltype(d)::value;
          auto kern = fw_kernel(epi, rev, [](auto e, auto r) { return tc_fw<T, D, decltype(r)::value, decltype(e)::value>; });
          return launch_fw(kern, p, g.ctas, FwSmem<D>::kBytes, false, pdl, st, mq, mk, mv, mh, mcs);
        });
    }
  });
}

struct BwWs {
  size_t off_states, off_h, off_n, off_m, total;
};
BwWs bw_ws(const mlstm_b200_shape& s) {
  BwWs w{};
  size_t tok = (size_t)s.B * s.NH * s.S, o = 0;
  w.off_states = o; o += align_up(tensor_states_bytes(s), 256);
  w.off_h = o; o += align_up(tok * s.DHHV * 2, 256);
  w.off_n = o; o += align_up(tok * 4, 256);
  w.off_m = o; o += align_up(tok * 4, 256);
  w.total = o;
  return w;
}

// ---------------------------------------------------------------------------------------------
// The backward of a head geometry with more than one block (tc_geometry) as square block problems.
//
// With n_out and every max state held constant (the definition of this backward, native/bw.py:44-47) every term
// of bw.py:106-203 is bilinear in (a bd-wide block of q / k, a bd-wide block of v / dh): dS = (dH V^T) . D and
// S = (Q K^T) . D are sums over column blocks, the state gradient dC (dqk x dv) splits into independent bd x bd
// blocks with the same decay, and the stabilisers depend on the gates only.  So a (DHQK, DHHV) problem is the sum of
// (DHQK / bd) x (DHHV / bd) tc_bw<bd> problems on strided views of the same tensors (no copies of q/k/v/dh;
// qk_scale = DHQK^-1/2 of the whole problem; each loads its block of the forward's saved states or recomputes it,
// bw.py:251-266).  dq / dk then take nv partials, dv nq and di / df nq nv.  The first partial of every output block
// is written in place, the others are added by the kernel that produces them (TMA reduce-add stores).
// bd x bd block (a, b) of a (BH, DK, DV) fp32 state <-> contiguous (BH, bd, bd); vec: (BH, DK) <-> (BH, bd)
__global__ void k_state_block(float* __restrict__ blk, float* __restrict__ full, int a, int b, int bd, int DK, int DV,
                              int64_t n, int scatter) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= n) return;
  const int64_t bh = idx / ((int64_t)bd * bd);
  const int r = (int)(idx / bd % bd), c = (int)(idx % bd);
  float* f = full + (bh * DK + a * bd + r) * DV + b * bd + c;
  if (scatter) *f = blk[idx]; else blk[idx] = *f;
}
__global__ void k_state_vec_block(float* __restrict__ blk, const float* __restrict__ full, int a, int bd, int DK, int64_t n) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= n) return;
  blk[idx] = full[(idx / bd) * DK + a * bd + idx % bd];
}
// Wide heads: di / df as the fp32 sum of the block problems' partials (part: [2][nparts][B NH S], di then df), rounded once
template <typename TO>
__global__ void k_sum_gate_partials(const TO* __restrict__ part, int nparts, int64_t n, int NH, int S, TO* di, int64_t di_sb,
                                    int64_t di_sh, int64_t di_ss, TO* df, int64_t df_sb, int64_t df_sh, int64_t df_ss) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= 2 * n) return;
  const int which = (int)(idx / n);
  const int64_t e = idx % n, bh = e / S, t = e % S, b = bh / NH, h = bh % NH;
  const TO* src = part + (int64_t)which * nparts * n + e;
  float acc = 0.f;
  for (int j = 0; j < nparts; ++j) acc += to_f32<TO>(src[(int64_t)j * n]);
  if (which == 0) di[b * di_sb + h * di_sh + t * di_ss] = from_f32<TO>(acc);
  else df[b * df_sb + h * df_sh + t * df_ss] = from_f32<TO>(acc);
}

// One bd x bd block problem of s; qk_scale stays that of the whole problem
mlstm_b200_shape block_shape(const mlstm_b200_shape& s, int bd) {
  mlstm_b200_shape b = s;
  b.DHQK = b.DHHV = bd;
  b.qk_scale = s.qk_scale > 0.f ? s.qk_scale : 1.f / sqrtf((float)s.DHQK);
  return b;
}
struct BlocksWs {
  size_t off_sub, sub_bytes, off_c0, off_n0, off_dcl, off_dc0, off_g, total;
};
BlocksWs blocks_ws(const mlstm_b200_shape& s, const TcGeometry& g) {
  BlocksWs w{};
  const size_t bh = (size_t)s.B * s.NH, bd = g.bd;
  size_t o = 0;
  w.sub_bytes = bw_ws(block_shape(s, g.bd)).total;
  w.off_sub = o; o += align_up(w.sub_bytes, 256);
  w.off_c0 = o; o += align_up(bh * bd * bd * 4, 256);
  w.off_n0 = o; o += align_up(bh * bd * 4, 256);
  w.off_dcl = o; o += align_up(bh * bd * bd * 4, 256);
  w.off_dc0 = o; o += align_up(bh * bd * bd * 4, 256);
  // gate_parts: the 16-bit di / df partial of every block problem, summed in fp32 by k_sum_gate_partials
  w.off_g = o;
  if (g.gate_parts) o += align_up(2 * (size_t)g.nq * g.nv * bh * s.S * 2, 256);
  w.total = o;
  return w;
}

// One tc_bw launch of a square problem (DHQK = DHHV = D).  c_states: the forward's saved states as nblocks D x D blocks per
// tile, of which this problem reads block `block`; NULL: recompute them into the workspace first (bw.py:251-266), as
// block 0 of 1.  acc_*: add into dq / dk, dv, di / df instead of overwriting them.
int bw_square(const mlstm_b200_bw_args& a, const void* c_states, int block, int nblocks, cudaStream_t st, int acc_qk,
              int acc_v, int acc_g) {
  const mlstm_b200_shape& s = a.shape;
  if (!c_states) {
    BwWs w = bw_ws(s);
    if (!a.workspace || a.workspace_bytes < w.total) {
      set_error("workspace too small: need %zu bytes, got %zu", w.total, a.workspace_bytes);
      return MLSTM_B200_EWORKSPACE;
    }
    char* ws = (char*)a.workspace;
    mlstm_b200_fw_args f{};
    f.shape = s;
    f.q = a.q; f.k = a.k; f.v = a.v; f.i = a.i; f.f = a.f;
    f.c_initial = a.c_initial; f.n_initial = a.n_initial; f.m_initial = a.m_initial;
    f.h.ptr = ws + w.off_h;
    f.h.stride[0] = (int64_t)s.NH * s.S * s.DHHV; f.h.stride[1] = (int64_t)s.S * s.DHHV; f.h.stride[2] = s.DHHV;
    f.h.stride[3] = 1;
    f.n_out = (float*)(ws + w.off_n); f.m_out = (float*)(ws + w.off_m);
    if (int e = run_fw(f, ws + w.off_states, st)) return e;
    c_states = ws + w.off_states;
    block = 0, nblocks = 1;
  }
  CUtensorMap mq, mk, mv, mdh, mcs, mdq, mdk, mdv;
  const int D = s.DHQK;
  mlstm_b200_shape sg = s;  // the gradients' tensor maps carry THEIR dtype (it matters for the reduce-add stores)
  if (s.grad_dtype) sg.dtype = s.grad_dtype;
  const bool mixed = sg.dtype != s.dtype;
  int r = make_map(&mq, a.q, s, D) | make_map(&mk, a.k, s, D) | make_map(&mv, a.v, s, D) | make_map(&mdh, a.dh, s, D) |
          make_states_map_blocks(&mcs, c_states, s, nblocks * D, D) | make_map(&mdq, a.dq, sg, D) |
          make_map(&mdk, a.dk, sg, D) | make_map(&mdv, a.dv, sg, D);
  if (r) {
    set_error("cuTensorMapEncodeTiled failed (%d)", r);
    return MLSTM_B200_ENODEVICE;
  }
  TcBwParams p{};
  set_gate_params(p, s, a.i, a.f);
  p.m0 = a.m_initial;
  p.n_out = a.n_out; p.m_out = a.m_out; p.dc_last = a.dc_last;
  p.di = a.di.ptr; p.di_sb = a.di.stride[0]; p.di_sh = a.di.stride[1]; p.di_ss = a.di.stride[2];
  p.df = a.df.ptr; p.df_sb = a.df.stride[0]; p.df_sh = a.df.stride[1]; p.df_ss = a.df.stride[2];
  p.dc0 = a.dc_initial;
  p.acc_qk = acc_qk; p.acc_v = acc_v; p.acc_g = acc_g;
  p.cs_rows = nblocks * D;
  p.cs_off = block * D;
  TC_SET_PROF(p, 4096);
  const int e = with_dtype(s.dtype, [&](auto t) {
    using T = decltype(t);
    using TX = std::conditional_t<std::is_same<T, __half>::value, __nv_bfloat16, __half>;  // the other 16-bit type
    return with_d32_64(D, [&](auto d) {
      constexpr int DD = decltype(d)::value;
      // mixed: kernel operands in one 16-bit dtype, gradients rounded once from fp32 to the other
      return mixed ? launch_bw<T, DD, TX>(p, mq, mk, mv, mdh, mcs, mdq, mdk, mdv, st)
                   : launch_bw<T, DD>(p, mq, mk, mv, mdh, mcs, mdq, mdk, mdv, st);
    });
  });
  if (e) return e;
  count_launch();
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

template <typename T>
int bw_by_blocks(const mlstm_b200_bw_args& a, const TcGeometry& g, cudaStream_t st) {
  const mlstm_b200_shape& s = a.shape;
  const BlocksWs w = blocks_ws(s, g);
  if (!a.workspace || a.workspace_bytes < w.total) {
    set_error("workspace too small: need %zu bytes, got %zu", w.total, a.workspace_bytes);
    return MLSTM_B200_EWORKSPACE;
  }
  char* ws = (char*)a.workspace;
  const int bd = g.bd, nq = g.nq, nv = g.nv;
  const int64_t bh = (int64_t)s.B * s.NH, nst = bh * bd * bd, nvec = bh * bd;
  auto cols = [&](const mlstm_b200_tensor& t, int j) {  // columns bd j .. bd j + bd - 1 of a wider tensor: a view
    mlstm_b200_tensor v = t;
    v.ptr = (char*)t.ptr + (size_t)j * bd * sizeof(T);
    return v;
  };
  auto state_block = [&](size_t off, const float* full, int qa, int vb, int scatter) {
    k_state_block<<<(unsigned)((nst + 255) / 256), 256, 0, st>>>((float*)(ws + off), (float*)full, qa, vb, bd, s.DHQK, s.DHHV,
                                                                  nst, scatter);
  };
  int launches = 0;
  bool first = true;
  const int64_t ntok = bh * s.S;
  auto gate_part = [&](int which, int j) {  // (B, NH, S) view of partial j of di (which = 0) or df (1)
    mlstm_b200_tensor t{};
    t.ptr = ws + w.off_g + ((size_t)which * nq * nv + j) * ntok * 2;
    t.stride[0] = (int64_t)s.NH * s.S; t.stride[1] = s.S; t.stride[2] = 1; t.stride[3] = 1;
    return t;
  };
  // With the forward's saved states (stored block-wise, make_states_map_blocks) every problem loads its block; without
  // them it recomputes its slice.
  const bool saved = a.c_states != nullptr;
  for (int qa = 0; qa < nq; ++qa) {
    for (int vb = 0; vb < nv; ++vb) {
      mlstm_b200_bw_args sub = a;
      sub.shape = block_shape(s, bd);
      sub.q = cols(a.q, qa); sub.k = cols(a.k, qa); sub.v = cols(a.v, vb); sub.dh = cols(a.dh, vb);
      sub.workspace = ws + w.off_sub; sub.workspace_bytes = w.sub_bytes;
      if (a.c_initial && !saved) {
        state_block(w.off_c0, a.c_initial, qa, vb, 0);
        k_state_vec_block<<<(unsigned)((nvec + 255) / 256), 256, 0, st>>>((float*)(ws + w.off_n0), a.n_initial, qa, bd, s.DHQK,
                                                                            nvec);
        sub.c_initial = (const float*)(ws + w.off_c0);
        sub.n_initial = (const float*)(ws + w.off_n0);
        launches += 2;
      }
      if (a.dc_last) {
        state_block(w.off_dcl, a.dc_last, qa, vb, 0);
        sub.dc_last = (const float*)(ws + w.off_dcl);
        ++launches;
      }
      if (a.dc_initial) sub.dc_initial = (float*)(ws + w.off_dc0);
      // The partial sums of an output block are added IN the kernel that produces the second one: dq_a, dk_a (sums over
      // the v blocks) and dv_b (sum over the qk blocks) through TMA reduce-add stores, di / df by their owner threads --
      // the block problems run one after the other on the stream, so the result is deterministic (one 16-bit rounding
      // per addition, as a separate accumulate pass would do) and no scratch copies or accumulate launches are needed.
      sub.dq = cols(a.dq, qa);
      sub.dk = cols(a.dk, qa);
      sub.dv = cols(a.dv, vb);
      sub.di = g.gate_parts ? gate_part(0, qa * nv + vb) : a.di;
      sub.df = g.gate_parts ? gate_part(1, qa * nv + vb) : a.df;
      if (int e = bw_square(sub, a.c_states, qa * nv + vb, nq * nv, st, vb > 0, qa > 0, !first && !g.gate_parts)) return e;
      if (a.dc_initial) {
        state_block(w.off_dc0, a.dc_initial, qa, vb, 1);
        ++launches;
      }
      first = false;
    }
  }
  if (g.gate_parts) {
    const unsigned grid = (unsigned)((2 * ntok + 255) / 256);
    with_dtype(s.grad_dtype ? s.grad_dtype : s.dtype, [&](auto t) {
      using TO = decltype(t);
      k_sum_gate_partials<TO><<<grid, 256, 0, st>>>((const TO*)(ws + w.off_g), nq * nv, ntok, s.NH, s.S, (TO*)a.di.ptr,
                                                    a.di.stride[0], a.di.stride[1], a.di.stride[2], (TO*)a.df.ptr,
                                                    a.df.stride[0], a.df.stride[1], a.df.stride[2]);
      return 0;
    });
    ++launches;
  }
  MLSTM_CUDA_CHECK(cudaGetLastError());
  count_launch(launches);  // the block problems counted their own launches
  return 0;
}

}  // namespace

// the views a call hands in can be described by TMA tensor maps (16-byte aligned base, 16-byte-multiple strides)
bool tensor_views_ok(const mlstm_b200_fw_args& a) {
  return tma_ok(a.q) && tma_ok(a.k) && tma_ok(a.v) && tma_ok(a.epilogue ? a.epilogue->y : a.h);
}
bool tensor_views_ok(const mlstm_b200_bw_args& a) {
  return tma_ok(a.q) && tma_ok(a.k) && tma_ok(a.v) && tma_ok(a.dh) && tma_ok(a.dq) && tma_ok(a.dk) && tma_ok(a.dv);
}

void tensor_set_clock_buffer(void* dev_ptr) {
#ifdef MLSTM_TC_PROFILE
  g_prof.store((long long*)dev_ptr);
#else
  (void)dev_ptr;
#endif
}
bool tensor_context_is_current() { return sm100_host::context_is_current(); }

bool tensor_supported(const mlstm_b200_shape& s) { return tc_geometry(s).fw != TcFw::none; }

size_t tensor_states_bytes(const mlstm_b200_shape& s) {
  if (!tensor_supported(s)) return 0;
  const size_t NT = (s.S + LT - 1) / LT;
  return (size_t)s.B * s.NH * NT * s.DHQK * s.DHHV * 2;
}

// forward needs no scratch; backward needs room to recompute the states when c_states is absent
size_t tensor_workspace_bytes(const mlstm_b200_shape& s, int backward) {
  if (!backward) return 256;
  const TcGeometry g = tc_geometry(s);
  return g.nq * g.nv > 1 ? blocks_ws(s, g).total : bw_ws(s).total;
}

int tensor_fw(const mlstm_b200_fw_args& a, cudaStream_t st) { return run_fw(a, a.c_states, st); }

// cudaOccupancyMaxActiveClusters of the forward with the fused epilogue in {2, 1, 1} clusters on the current device; 0 for
// a shape that does not launch it, -1 on a CUDA error
int tensor_fw_epilogue_clusters(const mlstm_b200_shape& s) {
  const TcGeometry g = tc_geometry(s);
  if (!g.cluster) return 0;
  auto query = [&](auto kern, int smem) {
    if (ensure_smem(kern, smem) != cudaSuccess) return -1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(g.ctas * s.B * s.NH), cfg.blockDim = dim3(kTcThreads), cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2, attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr, cfg.numAttrs = 1;
    int n = 0;
    return cudaOccupancyMaxActiveClusters(&n, kern, &cfg) == cudaSuccess ? n : -1;
  };
  return with_dtype(s.dtype, [&](auto t) {
    return with_d32_64(g.bd, [&](auto d) {
      constexpr int D = decltype(d)::value;
      return query(fw_rect_kernel<decltype(t), D>(true, s.reverse != 0), FwSmem<D>::kBytesPair);
    });
  });
}

int tensor_bw(const mlstm_b200_bw_args& a, cudaStream_t st) {
  if (!tensor_views_ok(a)) {
    set_error("tensor path needs 16-byte aligned q/k/v/dh/dq/dk/dv with strides that are multiples of 8 elements");
    return MLSTM_B200_EUNSUPPORTED;
  }
  const TcGeometry g = tc_geometry(a.shape);
  if (g.nq * g.nv == 1) return bw_square(a, a.c_states, 0, 1, st, 0, 0, 0);
  return with_dtype(a.shape.dtype, [&](auto t) { return bw_by_blocks<decltype(t)>(a, g, st); });
}

}  // namespace mlstm
