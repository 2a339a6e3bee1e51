// Exact-precision (fp32 FFMA) kernel family of the sm_100a mLSTM chunkwise path.
//
// This is the fp32 mode of the backend: all contractions are FFMA with fp32 accumulation so
// that fp32 inputs reproduce the reference within 1e-5 (a tcgen05 kind::tf32 path could not,
// SURVEY.md finding 9).  16-bit inputs are accepted too (loaded, widened, computed in fp32).
// The structure follows the math of SURVEY.md Appendix A, one kernel per reference stage:
//
//   k_states   inter-chunk C/n/m recurrence          native/fw.py:29-128     (also bw.py:251-266)
//   k_fw_h     intra-chunk outputs + combine         native/fw.py:131-221
//   k_bw_dc    state-gradient recurrence             native/bw.py:31-103
//   k_bw_dqkv  dQ/dK/dV (recomputed D, S) + dI       native/bw.py:106-203, 326
//   k_bw_df    whole-sequence reverse cumsum -> dF   native/bw.py:319-323
//
// h and the last states do not depend on the chunk length (the stabiliser m_t equals the
// step-recurrent one), so the kernels may run on an internal chunk that divides the requested
// one; it is chosen so that every tile fits in shared memory.
#include "common.cuh"

namespace mlstm {
namespace {

constexpr int kThreads = 256;

struct TView {  // strided tensor view in elements
  const void* ptr;
  int64_t sb, sh, ss;  // batch, head, token strides (innermost = 1)
};
struct GView {
  const void* ptr;
  int64_t sb, sh, ss;
};

struct ExactParams {
  int B, NH, S, DK, DV, L, NC;
  float eps, scale;
  TView q, k, v, dh;
  GView ig, fg;
  const float *c0, *n0, *m0;
  float *Cst, *Nst, *Mst;  // (BH, NC+1, DK, DV), (BH, NC+1, DK), (BH, NC+1)
  float* dCst;             // (BH, NC+1, DK, DV)
  float* acc;              // (BH, S): q.dq - k.dk
  void* h;                 // outputs
  int64_t h_sb, h_sh, h_ss;
  float *n_out, *m_out;
  float *c_last, *n_last, *m_last;
  const float *n_out_in, *m_out_in, *dc_last;
  void *dq, *dk, *dv, *di, *df;
  int64_t dq_s[3], dk_s[3], dv_s[3], di_s[3], df_s[3];
  float* dc0;
  int DVT;  // dv slice width of the recurrent kernels
  int DVB;  // v column block of k_fw_h / k_bw_dqkv (= DV when the whole of v fits in shared memory)
  int rev; // 1: anti-causal scan -- processing index t lives at memory token S-1-t (no data is moved)
  int sig;  // mlstm_b200_shape::siging: 1 sigmoid input gate, every max state 0; 2 the same without the normaliser
};
// memory token of processing index t, and the signed token step
__device__ __forceinline__ int64_t tok(const ExactParams& p, int64_t t) { return p.rev ? (int64_t)p.S - 1 - t : t; }
__device__ __forceinline__ int64_t sgn(const ExactParams& p) { return p.rev ? -1 : 1; }

// acc[a][j] += sum_k A(m_a, k) * B(k, n_j) with m_a = tm + a*MS, n_j = tn + j*NS.
// TA: A stored [k][m]; TB: B stored [n][k].  All leading dimensions are odd -> conflict-free.
template <bool TA, bool TB>
__device__ __forceinline__ void mm_tile(const float* __restrict__ A, int lda, const float* __restrict__ Bm, int ldb,
                                        int K, int tm, int MS, int tn, int NS, float (&acc)[4][4]) {
  for (int kk = 0; kk < K; ++kk) {
    float a[4], b[4];
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      a[x] = TA ? A[kk * lda + tm + x * MS] : A[(tm + x * MS) * lda + kk];
      b[x] = TB ? Bm[(tn + x * NS) * ldb + kk] : Bm[kk * ldb + tn + x * NS];
    }
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(a[x], b[y], acc[x][y]);
  }
}
__device__ __forceinline__ void zero_tile(float (&acc)[4][4]) {
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int y = 0; y < 4; ++y) acc[x][y] = 0.f;
}

template <typename T>
__device__ __forceinline__ void load_tile(float* dst, int ld, const T* src, int64_t row_stride, int rows, int cols) {
  for (int e = threadIdx.x; e < rows * cols; e += blockDim.x) {
    int r = e / cols, c = e - r * cols;
    dst[r * ld + c] = to_f32<T>(src[(int64_t)r * row_stride + c]);
  }
}

// -------------------------------------------------------------------------------------------
// k_states: sequential over chunks, one CTA per (b, h, dv-slice)
// -------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads) k_states(ExactParams p) {
  extern __shared__ float smem[];
  const int bh = blockIdx.x, b = bh / p.NH, hh = bh % p.NH;
  const int e0 = blockIdx.y * p.DVT;
  const int DVT = min(p.DVT, p.DV - e0);
  const int L = p.L, DK = p.DK, DV = p.DV;
  const int ldk = DK + 1, ldv = DVT | 1, ldc = DVT | 1;
  float* sK = smem;               // L x ldk
  float* sV = sK + L * ldk;       // L x ldv
  float* sC = sV + L * ldv;       // DK x ldc
  float* sN = sC + DK * ldc;      // DK
  float* sb = sN + DK;            // L
  float* si = sb + L;
  float* spm = si + L;
  float* sw = spm + L;
  __shared__ float s_g, s_amax;

  const T* kp = (const T*)p.k.ptr + b * p.k.sb + hh * p.k.sh;
  const T* vp = (const T*)p.v.ptr + b * p.v.sb + hh * p.v.sh + e0;
  const T* ip = (const T*)p.ig.ptr + b * p.ig.sb + hh * p.ig.sh;
  const T* fp = (const T*)p.fg.ptr + b * p.fg.sb + hh * p.fg.sh;

  for (int e = threadIdx.x; e < DK * DVT; e += blockDim.x) {
    int d = e / DVT, c = e - d * DVT;
    sC[d * ldc + c] = p.c0 ? p.c0[((int64_t)bh * DK + d) * DV + e0 + c] : 0.f;
  }
  for (int d = threadIdx.x; d < DK; d += blockDim.x) sN[d] = p.n0 ? p.n0[(int64_t)bh * DK + d] : 0.f;
  float m = p.m0 ? p.m0[bh] : 0.f;
  __syncthreads();

  const int MS = DK / 4, NS = DVT / 4;
  for (int j = 0; j <= p.NC; ++j) {
    // store the state entering chunk j (index NC = final state)
    float* Cd = p.Cst + ((int64_t)bh * (p.NC + 1) + j) * DK * DV;
    for (int e = threadIdx.x; e < DK * DVT; e += blockDim.x) {
      int d = e / DVT, c = e - d * DVT;
      Cd[(int64_t)d * DV + e0 + c] = sC[d * ldc + c];
    }
    if (blockIdx.y == 0) {
      for (int d = threadIdx.x; d < DK; d += blockDim.x) p.Nst[((int64_t)bh * (p.NC + 1) + j) * DK + d] = sN[d];
      if (threadIdx.x == 0) p.Mst[(int64_t)bh * (p.NC + 1) + j] = m;
    }
    if (j == p.NC) break;

    const int64_t m0 = tok(p, (int64_t)j * L), sg = sgn(p);
    load_tile<T>(sK, ldk, kp + m0 * p.k.ss, sg * p.k.ss, L, DK);
    load_tile<T>(sV, ldv, vp + m0 * p.v.ss, sg * p.v.ss, L, DVT);
    if (threadIdx.x < 32) {
      float amax;
      float g = chunk_gate_scan<T>(ip + m0 * p.ig.ss, sg * p.ig.ss, fp + m0 * p.fg.ss, sg * p.fg.ss, L, L, sb, si,
                                   spm, &amax, p.sig != 0);
      if (threadIdx.x == 0) { s_g = g; s_amax = amax; }
    }
    __syncthreads();
    const float g = s_g;
    const float m_next = p.sig ? 0.f : fmaxf(g + m, g + s_amax);  // fw.py:96-98
    const float decay = expf(g + m - m_next);             // fw.py:106
    for (int t = threadIdx.x; t < L; t += blockDim.x) sw[t] = expf(g - sb[t] + si[t] - m_next);  // fw.py:102
    __syncthreads();
    for (int e = threadIdx.x; e < L * DK; e += blockDim.x) {
      int t = e / DK, d = e - t * DK;
      sK[t * ldk + d] *= sw[t];
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < MS * NS; idx += blockDim.x) {
      int tm = idx / NS, tn = idx - tm * NS;
      float acc[4][4];
      zero_tile(acc);
      mm_tile<true, false>(sK, ldk, sV, ldv, L, tm, MS, tn, NS, acc);
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          float* c = &sC[(tm + x * MS) * ldc + tn + y * NS];
          *c = decay * *c + acc[x][y];
        }
    }
    for (int d = threadIdx.x; d < DK; d += blockDim.x) {
      float s = 0.f;
      for (int t = 0; t < L; ++t) s += sK[t * ldk + d];
      sN[d] = decay * sN[d] + s;  // fw.py:116
    }
    m = m_next;
    __syncthreads();
  }
  // last states (fw.py:302-309)
  if (p.c_last) {
    for (int e = threadIdx.x; e < DK * DVT; e += blockDim.x) {
      int d = e / DVT, c = e - d * DVT;
      p.c_last[((int64_t)bh * DK + d) * DV + e0 + c] = sC[d * ldc + c];
    }
    if (blockIdx.y == 0) {
      for (int d = threadIdx.x; d < DK; d += blockDim.x) p.n_last[(int64_t)bh * DK + d] = sN[d];
      if (threadIdx.x == 0) p.m_last[bh] = m;
    }
  }
}

// -------------------------------------------------------------------------------------------
// k_fw_h: one CTA per (chunk, b*h).  P and the denominators are computed once; h is then written in column blocks
// of width DVB, the V and C_{k-1} blocks taking turns in shared memory (one block when the whole of v fits).
// -------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads) k_fw_h(ExactParams p) {
  extern __shared__ float smem[];
  const int c = blockIdx.x, bh = blockIdx.y, b = bh / p.NH, hh = bh % p.NH;
  const int L = p.L, DK = p.DK, DV = p.DV, DVB = p.DVB;
  const int ldk = DK + 1, ldv = DVB + 1, ldp = L + 1;
  float* sQ = smem;
  float* sK = sQ + L * ldk;
  float* sV = sK + L * ldk;   // L x ldv: one column block of V
  float* sC = sV + L * ldv;   // DK x ldv: the same block of C_{k-1}
  float* sP = sC + DK * ldv;  // L x ldp
  float* sN = sP + L * ldp;   // DK
  float* sb = sN + DK;
  float* si = sb + L;
  float* spm = si + L;
  float* sbq = spm + L;   // bbar * scale
  float* sden = sbq + L;  // n_out + eps
  float* smt = sden + L;  // m_t

  const int64_t t0 = tok(p, (int64_t)c * L), sg = sgn(p);  // memory token of the chunk's first processed row
  load_tile<T>(sQ, ldk, (const T*)p.q.ptr + b * p.q.sb + hh * p.q.sh + t0 * p.q.ss, sg * p.q.ss, L, DK);
  load_tile<T>(sK, ldk, (const T*)p.k.ptr + b * p.k.sb + hh * p.k.sh + t0 * p.k.ss, sg * p.k.ss, L, DK);
  const T* vp = (const T*)p.v.ptr + b * p.v.sb + hh * p.v.sh + t0 * p.v.ss;
  const float* Cs = p.Cst + ((int64_t)bh * (p.NC + 1) + c) * DK * DV;
  load_tile<T>(sV, ldv, vp, sg * p.v.ss, L, DVB);  // column block 0
  load_tile<float>(sC, ldv, Cs, DV, DK, DVB);
  for (int d = threadIdx.x; d < DK; d += blockDim.x) sN[d] = p.Nst[((int64_t)bh * (p.NC + 1) + c) * DK + d];
  const float m_prev = p.Mst[(int64_t)bh * (p.NC + 1) + c];
  if (threadIdx.x < 32) {
    float amax;
    chunk_gate_scan<T>((const T*)p.ig.ptr + b * p.ig.sb + hh * p.ig.sh + t0 * p.ig.ss, sg * p.ig.ss,
                       (const T*)p.fg.ptr + b * p.fg.sb + hh * p.fg.sh + t0 * p.fg.ss, sg * p.fg.ss, L, L, sb, si, spm, &amax, p.sig != 0);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < L; t += blockDim.x)
    smt[t] = p.sig ? 0.f : sb[t] + fmaxf(m_prev, spm[t]);  // fw.py:178-184
  __syncthreads();

  {  // P = (Q K^T * scale) . D, fw.py:171-194
    const int MS = L / 4, NS = L / 4;
    for (int idx = threadIdx.x; idx < MS * NS; idx += blockDim.x) {
      int tm = idx / NS, tn = idx - tm * NS;
      float acc[4][4];
      zero_tile(acc);
      mm_tile<false, true>(sQ, ldk, sK, ldk, DK, tm, MS, tn, NS, acc);
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          int t = tm + x * MS, s = tn + y * NS;
          float d = (s <= t) ? expf(sb[t] - sb[s] + si[s] - smt[t]) : 0.f;
          sP[t * ldp + s] = acc[x][y] * p.scale * d;
        }
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < L; t += blockDim.x) {
    float rs = 0.f, qn = 0.f;
    for (int s = 0; s <= t; ++s) rs += sP[t * ldp + s];
    for (int d = 0; d < DK; ++d) qn = fmaf(sQ[t * ldk + d], sN[d], qn);
    float bq = expf(sb[t] + m_prev - smt[t]) * p.scale;  // fw.py:197-198
    float den = bq * qn + rs;                             // fw.py:204-206
    float nmax = fmaxf(fabsf(den), expf(-smt[t]));        // fw.py:208-210
    sbq[t] = bq;
    sden[t] = p.sig == 2 ? 1.f : nmax + p.eps;  // siging = 2: h is the numerator
    p.n_out[(int64_t)bh * p.S + t0 + sg * t] = nmax;  // saved vectors are indexed by memory token
    p.m_out[(int64_t)bh * p.S + t0 + sg * t] = smt[t];
  }
  __syncthreads();
  T* hp = (T*)p.h + b * p.h_sb + hh * p.h_sh + t0 * p.h_ss;
  for (int e0 = 0; e0 < DV; e0 += DVB) {  // h = (qbar C + P V) / (n + eps), fw.py:200-212
    const int W = min(DVB, DV - e0);
    if (e0) {
      __syncthreads();
      load_tile<T>(sV, ldv, vp + e0, sg * p.v.ss, L, W);
      load_tile<float>(sC, ldv, Cs + e0, DV, DK, W);
      __syncthreads();
    }
    const int MS = L / 4, NS = W / 4;
    for (int idx = threadIdx.x; idx < MS * NS; idx += blockDim.x) {
      int tm = idx / NS, tn = idx - tm * NS;
      float a1[4][4], a2[4][4];
      zero_tile(a1);
      zero_tile(a2);
      mm_tile<false, false>(sQ, ldk, sC, ldv, DK, tm, MS, tn, NS, a1);
      mm_tile<false, false>(sP, ldp, sV, ldv, L, tm, MS, tn, NS, a2);
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          int t = tm + x * MS, e = tn + y * NS;
          hp[(int64_t)t * sg * p.h_ss + e0 + e] = from_f32<T>((sbq[t] * a1[x][y] + a2[x][y]) / sden[t]);
        }
    }
  }
}

// -------------------------------------------------------------------------------------------
// k_bw_dc: reverse over chunks, one CTA per (b, h, dv-slice)
// -------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads) k_bw_dc(ExactParams p) {
  extern __shared__ float smem[];
  const int bh = blockIdx.x, b = bh / p.NH, hh = bh % p.NH;
  const int e0 = blockIdx.y * p.DVT;
  const int DVT = min(p.DVT, p.DV - e0);
  const int L = p.L, DK = p.DK, DV = p.DV;
  const int ldk = DK + 1, ldv = DVT | 1, ldc = DVT | 1;
  float* sQ = smem;
  float* sH = sQ + L * ldk;
  float* sC = sH + L * ldv;
  float* sb = sC + DK * ldc;
  float* si = sb + L;
  float* spm = si + L;
  __shared__ float s_g;

  const T* qp = (const T*)p.q.ptr + b * p.q.sb + hh * p.q.sh;
  const T* hp = (const T*)p.dh.ptr + b * p.dh.sb + hh * p.dh.sh + e0;
  const T* ip = (const T*)p.ig.ptr + b * p.ig.sb + hh * p.ig.sh;
  const T* fp = (const T*)p.fg.ptr + b * p.fg.sb + hh * p.fg.sh;

  for (int e = threadIdx.x; e < DK * DVT; e += blockDim.x) {
    int d = e / DVT, c = e - d * DVT;
    sC[d * ldc + c] = p.dc_last ? p.dc_last[((int64_t)bh * DK + d) * DV + e0 + c] : 0.f;
  }
  __syncthreads();
  const int MS = DK / 4, NS = DVT / 4;
  for (int j = p.NC; j >= 0; --j) {
    float* Cd = p.dCst + ((int64_t)bh * (p.NC + 1) + j) * DK * DV;
    for (int e = threadIdx.x; e < DK * DVT; e += blockDim.x) {
      int d = e / DVT, c = e - d * DVT;
      Cd[(int64_t)d * DV + e0 + c] = sC[d * ldc + c];
    }
    if (j == 0) break;
    const int c = j - 1;
    const int64_t t0 = tok(p, (int64_t)c * L), sg = sgn(p);
    load_tile<T>(sQ, ldk, qp + t0 * p.q.ss, sg * p.q.ss, L, DK);
    load_tile<T>(sH, ldv, hp + t0 * p.dh.ss, sg * p.dh.ss, L, DVT);
    if (threadIdx.x < 32) {
      float amax;
      float g = chunk_gate_scan<T>(ip + t0 * p.ig.ss, sg * p.ig.ss, fp + t0 * p.fg.ss, sg * p.fg.ss, L, L, sb, si, spm, &amax, p.sig != 0);
      if (threadIdx.x == 0) s_g = g;
    }
    __syncthreads();
    const float m_prev = p.Mst[(int64_t)bh * (p.NC + 1) + c], m_next = p.Mst[(int64_t)bh * (p.NC + 1) + c + 1];
    const float decay = expf(s_g + m_prev - m_next);  // bw.py:76
    for (int e = threadIdx.x; e < L * DK; e += blockDim.x) {
      int t = e / DK, d = e - t * DK;
      float bq = expf(sb[t] + m_prev - p.m_out_in[(int64_t)bh * p.S + t0 + sg * t]) * p.scale;  // bw.py:79-86
      sQ[t * ldk + d] *= bq;
    }
    if (p.sig != 2) {  // siging = 2: no normaliser, dh is used as it is
      for (int e = threadIdx.x; e < L * DVT; e += blockDim.x) {
        int t = e / DVT, x = e - t * DVT;
        sH[t * ldv + x] /= (p.n_out_in[(int64_t)bh * p.S + t0 + sg * t] + p.eps);  // bw.py:88-90
      }
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < MS * NS; idx += blockDim.x) {
      int tm = idx / NS, tn = idx - tm * NS;
      float acc[4][4];
      zero_tile(acc);
      mm_tile<true, false>(sQ, ldk, sH, ldv, L, tm, MS, tn, NS, acc);
#pragma unroll
      for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
          float* cc = &sC[(tm + x * MS) * ldc + tn + y * NS];
          *cc = decay * *cc + acc[x][y];  // bw.py:93-95
        }
    }
    __syncthreads();
  }
  if (p.dc0) {
    for (int e = threadIdx.x; e < DK * DVT; e += blockDim.x) {
      int d = e / DVT, c = e - d * DVT;
      p.dc0[((int64_t)bh * DK + d) * DV + e0 + c] = sC[d * ldc + c];
    }
  }
}

// -------------------------------------------------------------------------------------------
// k_bw_dqkv: one CTA per (chunk, b*h).  v is taken in column blocks of width DVB (one block when the whole of v
// fits in shared memory).  Each block writes its columns of dV and adds its part to dS and dI; every block but the
// last also adds its part of the inter-chunk terms of dK and dQ, which sum over v, to the accumulators sWk / sWq.
// The final dK / dQ passes add the last block's part, so one block needs neither the accumulators nor extra passes.
// -------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ int spart_width(int DK, int DVB) { return max(32, max(DK, DVB) / 4); }

__device__ __forceinline__ void load_acc(float (&acc)[4][4], const float* src, int ld, int tm, int MS, int tn, int NS) {
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int y = 0; y < 4; ++y) acc[x][y] = src[(tm + x * MS) * ld + tn + y * NS];
}
__device__ __forceinline__ void store_acc(const float (&acc)[4][4], float* dst, int ld, int tm, int MS, int tn, int NS) {
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int y = 0; y < 4; ++y) dst[(tm + x * MS) * ld + tn + y * NS] = acc[x][y];
}

template <typename T, bool kBlocked>  // kBlocked = false: DVB == DV, the loop below runs once
__global__ void __launch_bounds__(kThreads) k_bw_dqkv(ExactParams p) {
  extern __shared__ float smem[];
  const int c = blockIdx.x, bh = blockIdx.y, b = bh / p.NH, hh = bh % p.NH;
  const int L = p.L, DK = p.DK, DV = p.DV, DVB = p.DVB, nblk = kBlocked ? (DV + DVB - 1) / DVB : 1;
  const int ldk = DK + 1, ldv = DVB + 1, ldp = L + 1, spw = spart_width(DK, DVB);
  float* sQ = smem;
  float* sK = sQ + L * ldk;
  float* sV = sK + L * ldk;    // V block               L x ldv
  float* sH = sV + L * ldv;    // dH / (n + eps) block  L x ldv
  float* sC = sH + L * ldv;    // C_{k-1} block         DK x ldv
  float* sdC = sC + DK * ldv;  // dC_k block            DK x ldv
  float* sS = sdC + DK * ldv;  // Sbar      L x ldp
  float* sdS = sS + L * ldp;   // dS        L x ldp
  float* spart = sdS + L * ldp;  // L x spw row-dot partials
  float* sb = spart + L * spw;
  float* si = sb + L;
  float* spm = si + L;
  float* sab = spm + L;   // abar
  float* sbb = sab + L;   // bbar
  float* smt = sbb + L;   // m_out
  float* sacc = smt + L;  // q.dq - k.dk
  float* sWk = sacc + L;       // nblk > 1: V dC_k^T over the blocks before the last        L x ldk
  float* sWq = sWk + L * ldk;  // nblk > 1: dHt C_{k-1}^T over the blocks before the last  L x ldk
  float* sdi = sWq + L * ldk;  // nblk > 1: v . dv over the blocks before the last
  __shared__ float s_g;

  const int64_t t0 = tok(p, (int64_t)c * L), sg = sgn(p);
  const T* vp = (const T*)p.v.ptr + b * p.v.sb + hh * p.v.sh + t0 * p.v.ss;
  const T* dhp = (const T*)p.dh.ptr + b * p.dh.sb + hh * p.dh.sh + t0 * p.dh.ss;
  const float* Cs = p.Cst + ((int64_t)bh * (p.NC + 1) + c) * DK * DV;
  const float* dCs = p.dCst + ((int64_t)bh * (p.NC + 1) + c + 1) * DK * DV;
  auto load_block = [&](int e0, int W) {
    load_tile<T>(sV, ldv, vp + e0, sg * p.v.ss, L, W);
    load_tile<T>(sH, ldv, dhp + e0, sg * p.dh.ss, L, W);
    for (int e = threadIdx.x; e < DK * W; e += blockDim.x) {
      int d = e / W, x = e - d * W;
      sC[d * ldv + x] = Cs[(int64_t)d * DV + e0 + x];
      sdC[d * ldv + x] = dCs[(int64_t)d * DV + e0 + x];
    }
  };
  auto normalise_dh = [&](int W) {  // bw.py:135; siging = 2: no normaliser, dh is used as it is
    if (p.sig == 2) return;
    for (int e = threadIdx.x; e < L * W; e += blockDim.x) {
      int t = e / W, x = e - t * W;
      sH[t * ldv + x] /= (p.n_out_in[(int64_t)bh * p.S + t0 + sg * t] + p.eps);
    }
  };
  load_tile<T>(sQ, ldk, (const T*)p.q.ptr + b * p.q.sb + hh * p.q.sh + t0 * p.q.ss, sg * p.q.ss, L, DK);
  load_tile<T>(sK, ldk, (const T*)p.k.ptr + b * p.k.sb + hh * p.k.sh + t0 * p.k.ss, sg * p.k.ss, L, DK);
  load_block(0, DVB);
  if (threadIdx.x < 32) {
    float amax;
    float g = chunk_gate_scan<T>((const T*)p.ig.ptr + b * p.ig.sb + hh * p.ig.sh + t0 * p.ig.ss, sg * p.ig.ss,
                                 (const T*)p.fg.ptr + b * p.fg.sb + hh * p.fg.sh + t0 * p.fg.ss, sg * p.fg.ss, L, L, sb, si,
                                 spm, &amax, p.sig != 0);
    if (threadIdx.x == 0) s_g = g;
  }
  __syncthreads();
  const float m_prev = p.Mst[(int64_t)bh * (p.NC + 1) + c], m_next = p.Mst[(int64_t)bh * (p.NC + 1) + c + 1];
  for (int t = threadIdx.x; t < L; t += blockDim.x) {
    float mt = p.m_out_in[(int64_t)bh * p.S + t0 + sg * t];
    smt[t] = mt;
    sab[t] = expf(s_g - sb[t] + si[t] - m_next);  // bw.py:181,187
    sbb[t] = expf(sb[t] + m_prev - mt);           // bw.py:186
  }
  normalise_dh(DVB);
  __syncthreads();

  const int64_t tok0 = (int64_t)bh * p.S + (int64_t)c * L;  // the q.dq - k.dk workspace is in processing order
  T* dvp = (T*)p.dv + b * p.dv_s[0] + hh * p.dv_s[1] + t0 * p.dv_s[2];
  T* dip = (T*)p.di + b * p.di_s[0] + hh * p.di_s[1] + t0 * p.di_s[2];
  int e0 = 0, W = DVB;  // the block in shared memory: columns [e0, e0 + W)
  for (int blk = 0; blk < nblk; ++blk) {
    const bool last = blk == nblk - 1;
    if (blk) {
      e0 += DVB;
      W = min(DVB, DV - e0);
      __syncthreads();
      load_block(e0, W);
      __syncthreads();
      normalise_dh(W);
      __syncthreads();
    }
    {  // Sbar (first block) and dS (summed over the blocks, times D after the last), bw.py:153-167
      const int MS = L / 4, NS = L / 4;
      for (int idx = threadIdx.x; idx < MS * NS; idx += blockDim.x) {
        int tm = idx / NS, tn = idx - tm * NS;
        float a1[4][4], a2[4][4];
        zero_tile(a1);
        if (blk) load_acc(a2, sdS, ldp, tm, MS, tn, NS);
        else zero_tile(a2);
        if (!blk) mm_tile<false, true>(sQ, ldk, sK, ldk, DK, tm, MS, tn, NS, a1);
        mm_tile<false, true>(sH, ldv, sV, ldv, W, tm, MS, tn, NS, a2);
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y) {
            int t = tm + x * MS, s = tn + y * NS;
            float d = (s <= t && (!blk || last)) ? expf(sb[t] - sb[s] + si[s] - smt[t]) : 0.f;
            if (!blk) sS[t * ldp + s] = a1[x][y] * p.scale * d;
            sdS[t * ldp + s] = last ? a2[x][y] * d : a2[x][y];
          }
      }
    }
    __syncthreads();
    {  // dV = Sbar^T dHt + abar (K dC_k); dI = v . dv   (bw.py:164,190,326)
      const int MS = L / 4, NS = W / 4;
      for (int idx0 = 0; idx0 < MS * NS; idx0 += blockDim.x) {
        int idx = idx0 + threadIdx.x;
        if (idx < MS * NS) {
          int tm = idx / NS, tn = idx - tm * NS;
          float a1[4][4], a2[4][4];
          zero_tile(a1);
          zero_tile(a2);
          mm_tile<true, false>(sS, ldp, sH, ldv, L, tm, MS, tn, NS, a1);
          mm_tile<false, false>(sK, ldk, sdC, ldv, DK, tm, MS, tn, NS, a2);
#pragma unroll
          for (int x = 0; x < 4; ++x) {
            int s = tm + x * MS;
            float part = 0.f;
#pragma unroll
            for (int y = 0; y < 4; ++y) {
              int e = tn + y * NS;
              float val = a1[x][y] + sab[s] * a2[x][y];
              dvp[(int64_t)s * sg * p.dv_s[2] + e0 + e] = from_f32<T>(val);
              part = fmaf(sV[s * ldv + e], val, part);
            }
            spart[s * spw + tn] = part;
          }
        }
      }
      __syncthreads();
      for (int s = threadIdx.x; s < L; s += blockDim.x) {
        float r = blk ? sdi[s] : 0.f;
        for (int x = 0; x < NS; ++x) r += spart[s * spw + x];
        if (!last) {
          sdi[s] = r;
          continue;
        }
        if (p.sig) r *= 1.f - expf(si[s]);  // d logsigmoid(i)/di = sigmoid(-i) = 1 - exp(logsigmoid(i))
        dip[(int64_t)s * sg * p.di_s[2]] = from_f32<T>(r);
      }
    }
    if (!last) {  // this block's part of V dC_k^T and dHt C_{k-1}^T
      const int MS = L / 4, NS = DK / 4;
      for (int idx = threadIdx.x; idx < MS * NS; idx += blockDim.x) {
        int tm = idx / NS, tn = idx - tm * NS;
        float a1[4][4], a2[4][4];
        if (blk) {
          load_acc(a1, sWk, ldk, tm, MS, tn, NS);
          load_acc(a2, sWq, ldk, tm, MS, tn, NS);
        } else {
          zero_tile(a1);
          zero_tile(a2);
        }
        mm_tile<false, true>(sV, ldv, sdC, ldv, W, tm, MS, tn, NS, a1);
        mm_tile<false, true>(sH, ldv, sC, ldv, W, tm, MS, tn, NS, a2);
        store_acc(a1, sWk, ldk, tm, MS, tn, NS);
        store_acc(a2, sWq, ldk, tm, MS, tn, NS);
      }
    }
  }
  __syncthreads();
  {  // dK = scale dS^T Q + abar (V dC_k^T)   (bw.py:170,192)
    const int MS = L / 4, NS = DK / 4;
    T* op = (T*)p.dk + b * p.dk_s[0] + hh * p.dk_s[1] + t0 * p.dk_s[2];
    for (int idx0 = 0; idx0 < MS * NS; idx0 += blockDim.x) {
      int idx = idx0 + threadIdx.x;
      if (idx < MS * NS) {
        int tm = idx / NS, tn = idx - tm * NS;
        float a1[4][4], a2[4][4];
        zero_tile(a1);
        if (nblk > 1) load_acc(a2, sWk, ldk, tm, MS, tn, NS);
        else zero_tile(a2);
        mm_tile<true, false>(sdS, ldp, sQ, ldk, L, tm, MS, tn, NS, a1);
        mm_tile<false, true>(sV, ldv, sdC, ldv, W, tm, MS, tn, NS, a2);
#pragma unroll
        for (int x = 0; x < 4; ++x) {
          int s = tm + x * MS;
          float part = 0.f;
#pragma unroll
          for (int y = 0; y < 4; ++y) {
            int d = tn + y * NS;
            float val = p.scale * a1[x][y] + sab[s] * a2[x][y];
            op[(int64_t)s * sg * p.dk_s[2] + d] = from_f32<T>(val);
            part = fmaf(sK[s * ldk + d], val, part);
          }
          spart[s * spw + tn] = part;
        }
      }
    }
    __syncthreads();
    for (int s = threadIdx.x; s < L; s += blockDim.x) {
      float r = 0.f;
      for (int x = 0; x < NS; ++x) r += spart[s * spw + x];
      sacc[s] = -r;
    }
    __syncthreads();
  }
  {  // dQ = scale dS K + scale bbar (dHt C_{k-1}^T)   (bw.py:169,193)
    const int MS = L / 4, NS = DK / 4;
    T* op = (T*)p.dq + b * p.dq_s[0] + hh * p.dq_s[1] + t0 * p.dq_s[2];
    for (int idx0 = 0; idx0 < MS * NS; idx0 += blockDim.x) {
      int idx = idx0 + threadIdx.x;
      if (idx < MS * NS) {
        int tm = idx / NS, tn = idx - tm * NS;
        float a1[4][4], a2[4][4];
        zero_tile(a1);
        if (nblk > 1) load_acc(a2, sWq, ldk, tm, MS, tn, NS);
        else zero_tile(a2);
        mm_tile<false, false>(sdS, ldp, sK, ldk, L, tm, MS, tn, NS, a1);
        mm_tile<false, true>(sH, ldv, sC, ldv, W, tm, MS, tn, NS, a2);
#pragma unroll
        for (int x = 0; x < 4; ++x) {
          int t = tm + x * MS;
          float part = 0.f;
#pragma unroll
          for (int y = 0; y < 4; ++y) {
            int d = tn + y * NS;
            float val = p.scale * (a1[x][y] + sbb[t] * a2[x][y]);
            op[(int64_t)t * sg * p.dq_s[2] + d] = from_f32<T>(val);
            part = fmaf(sQ[t * ldk + d], val, part);
          }
          spart[t * spw + tn] = part;
        }
      }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < L; t += blockDim.x) {
      float r = 0.f;
      for (int x = 0; x < NS; ++x) r += spart[t * spw + x];
      p.acc[tok0 + t] = r + sacc[t];  // q.dq - k.dk, bw.py:321
    }
  }
}

// -------------------------------------------------------------------------------------------
// k_bw_df: dF_t = sigmoid(-f_t) * sum_{tau >= t} acc_tau, one warp per (b, h)   (bw.py:321-323)
// -------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_bw_df(ExactParams p) {
  const int bh = blockIdx.x, b = bh / p.NH, hh = bh % p.NH, lane = threadIdx.x;
  const float* acc = p.acc + (int64_t)bh * p.S;
  const T* fp = (const T*)p.fg.ptr + b * p.fg.sb + hh * p.fg.sh;
  T* dfp = (T*)p.df + b * p.df_s[0] + hh * p.df_s[1];
  float carry = 0.f;
  for (int base = p.S - 32; base > -32; base -= 32) {
    int t = base + lane;
    float v = (t >= 0) ? acc[t] : 0.f;
    // inclusive suffix sum within the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      float u = __shfl_down_sync(0xffffffffu, v, o);
      if (lane + o < 32) v += u;
    }
    v += carry;
    if (t >= 0) {
      const int64_t mt = tok(p, t);
      dfp[mt * p.df_s[2]] = from_f32<T>(v * sigmoid_neg_f32(to_f32<T>(fp[mt * p.fg.ss])));
    }
    carry = __shfl_sync(0xffffffffu, v, 0);
  }
}

// -------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------
// Dynamic shared memory a CTA may use: the 227 KB per-block limit less the kernels' static __shared__ scalars.
constexpr size_t kMaxSmem = 227 * 1024 - 128;

size_t smem_states(int L, int DK, int DVT) {
  return sizeof(float) * ((size_t)L * (DK + 1) + (size_t)L * (DVT | 1) + (size_t)DK * (DVT | 1) + DK + 4 * L);
}
size_t smem_fw_h(int L, int DK, int DVB) {
  return sizeof(float) * ((size_t)2 * L * (DK + 1) + (size_t)L * (DVB + 1) + (size_t)DK * (DVB + 1) +
                          (size_t)L * (L + 1) + DK + 6 * L);
}
size_t smem_bw_dc(int L, int DK, int DVT) {
  return sizeof(float) * ((size_t)L * (DK + 1) + (size_t)L * (DVT | 1) + (size_t)DK * (DVT | 1) + 3 * L);
}
size_t smem_bw_dqkv(int L, int DK, int DV, int DVB) {
  size_t n = (size_t)2 * L * (DK + 1) + (size_t)2 * L * (DVB + 1) + (size_t)2 * DK * (DVB + 1) + (size_t)2 * L * (L + 1) +
             (size_t)L * spart_width(DK, DVB) + 7 * L;
  if (DVB < DV) n += (size_t)2 * L * (DK + 1) + L;  // the accumulators over the v blocks
  return sizeof(float) * n;
}

constexpr int kMaxDK = 256, kMaxDV = 512;

// v column block of k_fw_h (backward = 0) or k_bw_dqkv (1) at internal chunk L: the widest that fits in shared
// memory, from splitting v into as few near-equal blocks of a multiple of 4 columns as possible; 0 if none fits.
int pick_dvb(int L, int DK, int DV, int backward) {
  for (int n = 1; n <= DV / 4; ++n) {
    const int dvb = ((DV + n - 1) / n + 3) & ~3;
    if ((backward ? smem_bw_dqkv(L, DK, DV, dvb) : smem_fw_h(L, DK, dvb)) <= kMaxSmem) return dvb;
  }
  return 0;
}

// Largest internal chunk (dividing the requested one) whose tiles fit in shared memory.  A chunk that keeps the
// whole of v resident in both kernels is preferred over a larger one that needs v blocks.
int pick_chunk(const mlstm_b200_shape& s) {
  if ((s.DHQK & 3) || (s.DHHV & 3) || s.DHQK > kMaxDK || s.DHHV > kMaxDV) return 0;
  for (int blocked = 0; blocked < 2; ++blocked) {
    for (int L = s.chunk_size < 64 ? s.chunk_size : 64; L >= 4; --L) {
      if ((s.chunk_size % L) || (L & 3)) continue;
      const int fw = pick_dvb(L, s.DHQK, s.DHHV, 0), bw = pick_dvb(L, s.DHQK, s.DHHV, 1);
      if (fw && bw && (blocked || (fw == s.DHHV && bw == s.DHHV))) return L;
    }
  }
  return 0;
}

int check_shape(const mlstm_b200_shape& s) {
  if (s.B <= 0 || s.NH <= 0 || s.S <= 0 || s.DHQK <= 0 || s.DHHV <= 0 || s.chunk_size <= 0) {
    set_error("non-positive dimension");
    return MLSTM_B200_EINVAL;
  }
  if (s.S % s.chunk_size) {
    set_error("Sequence length %d is not divisible by chunk size %d.", s.S, s.chunk_size);
    return MLSTM_B200_EINVAL;
  }
  if ((s.DHQK & 3) || (s.DHHV & 3) || s.DHQK > kMaxDK || s.DHHV > kMaxDV) {
    set_error("exact path needs head dims that are multiples of 4 with DHQK <= %d and DHHV <= %d (got %d, %d)", kMaxDK,
              kMaxDV, s.DHQK, s.DHHV);
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (pick_chunk(s) == 0) {
    set_error("exact path: no internal chunk size fits shared memory for chunk=%d DHQK=%d DHHV=%d", s.chunk_size,
              s.DHQK, s.DHHV);
    return MLSTM_B200_EUNSUPPORTED;
  }
  return 0;
}

struct WsLayout {
  size_t off_C, off_N, off_M, off_dC, off_acc, total;
};
WsLayout ws_layout(const mlstm_b200_shape& s, int L, int backward) {
  WsLayout w{};
  size_t BH = (size_t)s.B * s.NH, NC1 = s.S / L + 1;
  size_t o = 0;
  w.off_C = o;
  o += align_up(BH * NC1 * s.DHQK * s.DHHV * sizeof(float), 256);
  w.off_N = o;
  o += align_up(BH * NC1 * s.DHQK * sizeof(float), 256);
  w.off_M = o;
  o += align_up(BH * NC1 * sizeof(float), 256);
  if (backward) {
    w.off_dC = o;
    o += align_up(BH * NC1 * s.DHQK * s.DHHV * sizeof(float), 256);
    w.off_acc = o;
    o += align_up(BH * s.S * sizeof(float), 256);
  }
  w.total = o;
  return w;
}

TView tview(const mlstm_b200_tensor& t) { return TView{t.ptr, t.stride[0], t.stride[1], t.stride[2]}; }
GView gview(const mlstm_b200_tensor& t) { return GView{t.ptr, t.stride[0], t.stride[1], t.stride[2]}; }

template <typename K>
int set_smem(K kernel, size_t bytes) {
  MLSTM_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

int pick_dvt(const mlstm_b200_shape& s, int L) {
  // slice dv so that the sequential kernels expose more CTAs and their tiles fit in shared memory; keep slices
  // multiples of 4 (the last one may be narrower)
  auto fits = [&](int d) { return smem_states(L, s.DHQK, d) <= kMaxSmem && smem_bw_dc(L, s.DHQK, d) <= kMaxSmem; };
  int dvt = s.DHHV;
  while (dvt > 16 && (dvt % 8) == 0 && ((long)s.B * s.NH * (s.DHHV / dvt) < 592 || !fits(dvt))) dvt /= 2;
  while (!fits(dvt)) dvt = (dvt / 2 + 3) & ~3;
  return dvt;
}

template <typename T>
int launch_states(ExactParams& p, cudaStream_t st) {
  size_t sm = smem_states(p.L, p.DK, p.DVT);
  if (int e = set_smem(k_states<T>, sm)) return e;
  dim3 grid(p.B * p.NH, (p.DV + p.DVT - 1) / p.DVT);
  k_states<T><<<grid, kThreads, sm, st>>>(p);
  count_launch();
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

size_t exact_workspace_bytes(const mlstm_b200_shape& s, int backward) {
  int L = pick_chunk(s);
  if (L == 0) return 0;
  return ws_layout(s, L, backward).total;
}

int exact_fw(const mlstm_b200_fw_args& a, cudaStream_t st) {
  const mlstm_b200_shape& s = a.shape;
  if (int e = check_shape(s)) return e;
  const int L = pick_chunk(s);
  WsLayout w = ws_layout(s, L, 0);
  if (a.workspace_bytes < w.total || !a.workspace) {
    set_error("workspace too small: need %zu bytes, got %zu", w.total, a.workspace_bytes);
    return MLSTM_B200_EWORKSPACE;
  }
  ExactParams p{};
  p.B = s.B; p.NH = s.NH; p.S = s.S; p.DK = s.DHQK; p.DV = s.DHHV; p.L = L; p.NC = s.S / L;
  p.eps = s.eps;
  p.scale = s.qk_scale > 0.f ? s.qk_scale : 1.f / sqrtf((float)s.DHQK);
  p.q = tview(a.q); p.k = tview(a.k); p.v = tview(a.v);
  p.ig = gview(a.i); p.fg = gview(a.f);
  p.c0 = a.c_initial; p.n0 = a.n_initial; p.m0 = a.m_initial;
  char* ws = (char*)a.workspace;
  p.Cst = (float*)(ws + w.off_C); p.Nst = (float*)(ws + w.off_N); p.Mst = (float*)(ws + w.off_M);
  p.h = a.h.ptr; p.h_sb = a.h.stride[0]; p.h_sh = a.h.stride[1]; p.h_ss = a.h.stride[2];
  p.n_out = a.n_out; p.m_out = a.m_out;
  p.c_last = a.c_last; p.n_last = a.n_last; p.m_last = a.m_last;
  p.DVT = pick_dvt(s, L);
  p.DVB = pick_dvb(L, p.DK, p.DV, 0);
  p.rev = s.reverse ? 1 : 0;
  p.sig = s.siging;  // 0, 1 or 2 (checked at the C-ABI)
  MLSTM_DISPATCH_DTYPE(s.dtype, T, {
    if (int e = launch_states<T>(p, st)) return e;
    size_t sm = smem_fw_h(L, p.DK, p.DVB);
    if (int e = set_smem(k_fw_h<T>, sm)) return e;
    k_fw_h<T><<<dim3(p.NC, p.B * p.NH), kThreads, sm, st>>>(p);
    count_launch();
    MLSTM_CUDA_CHECK(cudaGetLastError());
  });
  return 0;
}

int exact_bw(const mlstm_b200_bw_args& a, cudaStream_t st) {
  const mlstm_b200_shape& s = a.shape;
  if (int e = check_shape(s)) return e;
  const int L = pick_chunk(s);
  WsLayout w = ws_layout(s, L, 1);
  if (a.workspace_bytes < w.total || !a.workspace) {
    set_error("workspace too small: need %zu bytes, got %zu", w.total, a.workspace_bytes);
    return MLSTM_B200_EWORKSPACE;
  }
  ExactParams p{};
  p.B = s.B; p.NH = s.NH; p.S = s.S; p.DK = s.DHQK; p.DV = s.DHHV; p.L = L; p.NC = s.S / L;
  p.eps = s.eps;
  p.scale = s.qk_scale > 0.f ? s.qk_scale : 1.f / sqrtf((float)s.DHQK);
  p.q = tview(a.q); p.k = tview(a.k); p.v = tview(a.v); p.dh = tview(a.dh);
  p.ig = gview(a.i); p.fg = gview(a.f);
  p.c0 = a.c_initial; p.n0 = a.n_initial; p.m0 = a.m_initial;
  char* ws = (char*)a.workspace;
  p.Cst = (float*)(ws + w.off_C); p.Nst = (float*)(ws + w.off_N); p.Mst = (float*)(ws + w.off_M);
  p.dCst = (float*)(ws + w.off_dC); p.acc = (float*)(ws + w.off_acc);
  p.n_out_in = a.n_out; p.m_out_in = a.m_out; p.dc_last = a.dc_last;
  p.dq = a.dq.ptr; p.dk = a.dk.ptr; p.dv = a.dv.ptr; p.di = a.di.ptr; p.df = a.df.ptr;
  for (int x = 0; x < 3; ++x) {
    p.dq_s[x] = a.dq.stride[x]; p.dk_s[x] = a.dk.stride[x]; p.dv_s[x] = a.dv.stride[x];
    p.di_s[x] = a.di.stride[x]; p.df_s[x] = a.df.stride[x];
  }
  p.dc0 = a.dc_initial;
  p.DVT = pick_dvt(s, L);
  p.DVB = pick_dvb(L, p.DK, p.DV, 1);
  p.rev = s.reverse ? 1 : 0;
  p.sig = s.siging;  // 0, 1 or 2 (checked at the C-ABI)
  MLSTM_DISPATCH_DTYPE(s.dtype, T, {
    if (int e = launch_states<T>(p, st)) return e;  // recompute C/n/m states (bw.py:251-266)
    size_t sm = smem_bw_dc(L, p.DK, p.DVT);
    if (int e = set_smem(k_bw_dc<T>, sm)) return e;
    k_bw_dc<T><<<dim3(p.B * p.NH, (p.DV + p.DVT - 1) / p.DVT), kThreads, sm, st>>>(p);
    count_launch();
    MLSTM_CUDA_CHECK(cudaGetLastError());
    sm = smem_bw_dqkv(L, p.DK, p.DV, p.DVB);
    auto dqkv = p.DVB < p.DV ? k_bw_dqkv<T, true> : k_bw_dqkv<T, false>;
    if (int e = set_smem(dqkv, sm)) return e;
    dqkv<<<dim3(p.NC, p.B * p.NH), kThreads, sm, st>>>(p);
    count_launch();
    MLSTM_CUDA_CHECK(cudaGetLastError());
    k_bw_df<T><<<p.B * p.NH, 32, 0, st>>>(p);
    count_launch();
    MLSTM_CUDA_CHECK(cudaGetLastError());
  });
  return 0;
}

}  // namespace mlstm
