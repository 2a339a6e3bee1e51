// Recurrent (token-by-token) mLSTM: the step kernel and the sequence loop around it (SURVEY.md section 8(f) #4).
// Reference: mlstm_recurrent_step__native_fw, mlstm_kernels/torch/recurrent/native_step.py:8-101, and the loop
// _mlstm_recurrent_sequence_loop_fw, recurrent/native_sequence.py:14-130 -- what the reference's inference wrapper
// (wrap_chunkwise__arbitrary_sequence_length, kernel_wrappers.py:12-201) runs for the tokens that do not fill a
// chunk, and what generation-style callers run one token at a time.
//
// One CTA of 256 threads per (batch, head) keeps the state ON CHIP for the whole call: C (DHQK x DHHV fp32) in
// registers -- a thread owns DHQK / TPC rows of one column, TPC = 256 / DHHV adjacent lanes share a column so that
// the q . C column sums close with two or three shuffles -- n in shared memory, m in a register.  A single step
// (S = 1) is HBM-bound on reading and writing C once (8 B per state element); a sequence of S steps moves the state
// once instead of S times, which is the point of having the loop inside the kernel.  No tensor cores: a step is a
// rank-1 update plus a matrix-vector product.
#include "common.cuh"

namespace mlstm {
namespace {

constexpr int kStepThreads = 256;

template <typename T>
__device__ __forceinline__ float round_to(float x) { return to_f32<T>(from_f32<T>(x)); }

struct StepParams {
  int B, NH, S, siging;  // mlstm_b200_recurrent_args::siging: 0, 1 or 2 (no normaliser)
  float eps, scale;
  const void *q, *k, *v, *ig, *fg;
  int64_t q_sb, q_sh, q_ss, k_sb, k_sh, k_ss, v_sb, v_sh, v_ss, i_sb, i_sh, i_ss, f_sb, f_sh, f_ss;
  void* h;
  int64_t h_sb, h_sh, h_ss;
  const float *c0, *n0, *m0;
  float *c1, *n1, *m1;
};

template <typename T, int DK, int DV>
__global__ void __launch_bounds__(kStepThreads) k_recurrent(StepParams p) {
  constexpr int TPC = kStepThreads / DV;  // threads per column of C
  constexpr int RPT = DK / TPC;           // rows of that column per thread
  static_assert(TPC >= 2 && TPC <= 8 && RPT >= 1, "geometry");
  __shared__ float sq[DK], sk[DK], sv[DV], sn[DK], s_red[8], s_gate[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int bh = blockIdx.x, b = bh / p.NH, hd = bh % p.NH;
  const int j = tid / TPC, rg = tid % TPC;  // column of C, row group: rows rg, rg + TPC, ...

  float C[RPT];
  if (p.c0) {
    const float* src = p.c0 + (int64_t)bh * DK * DV;
#pragma unroll
    for (int r = 0; r < RPT; ++r) C[r] = src[(int64_t)(rg + r * TPC) * DV + j];
  } else {
#pragma unroll
    for (int r = 0; r < RPT; ++r) C[r] = 0.f;
  }
  if (tid < DK) sn[tid] = p.n0 ? p.n0[(int64_t)bh * DK + tid] : 0.f;
  float m = p.m0 ? p.m0[bh] : 0.f;

  const T* qp = (const T*)p.q + b * p.q_sb + hd * p.q_sh;
  const T* kp = (const T*)p.k + b * p.k_sb + hd * p.k_sh;
  const T* vp = (const T*)p.v + b * p.v_sb + hd * p.v_sh;
  const T* ip = (const T*)p.ig + b * p.i_sb + hd * p.i_sh;
  const T* fp = (const T*)p.fg + b * p.f_sb + hd * p.f_sh;
  T* hp = (T*)p.h + b * p.h_sb + hd * p.h_sh;

  for (int t = 0; t < p.S; ++t) {
    __syncthreads();  // the previous step's readers of sq / sk / sv / s_red are done
    if (tid < DK) {
      // vecQ_scaled = vecQ * DHQK^-0.5 in the q/k/v dtype (native_step.py:74)
      sq[tid] = round_to<T>(to_f32<T>(qp[(int64_t)t * p.q_ss + tid]) * p.scale);
      sk[tid] = to_f32<T>(kp[(int64_t)t * p.k_ss + tid]);
    }
    if (tid >= kStepThreads - DV) sv[tid - (kStepThreads - DV)] = to_f32<T>(vp[(int64_t)t * p.v_ss + tid - (kStepThreads - DV)]);
    if (tid == 0) {
      s_gate[0] = to_f32<T>(ip[(int64_t)t * p.i_ss]);
      s_gate[1] = to_f32<T>(fp[(int64_t)t * p.f_ss]);
    }
    __syncthreads();
    // gates and stabiliser (native_step.py:64-72); sigmoid input gate: i <- logsigmoid(i), no max state
    float ig = s_gate[0];
    const float lf = logsigmoid_f32(s_gate[1]);
    float m_new;
    if (p.siging) {
      ig = logsigmoid_f32(ig);
      m_new = 0.f;
    } else {
      m_new = fmaxf(lf + m, ig);
    }
    const float fa = expf(lf + m - m_new), ia = expf(ig - m_new);
    // C_t = f C_{t-1} + i k v^T; numerator q C_t with C_t rounded to the q/k/v dtype (native_step.py:75-81)
    const float iv = ia * sv[j];
    float acc = 0.f;
#pragma unroll
    for (int r = 0; r < RPT; ++r) {
      const int d = rg + r * TPC;
      C[r] = fa * C[r] + iv * sk[d];
      acc += sq[d] * round_to<T>(C[r]);
    }
#pragma unroll
    for (int o = 1; o < TPC; o <<= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    // n_t = f n_{t-1} + i k (native_step.py:78); q . n_t (native_step.py:84-87)
    float part = 0.f;
    if (tid < DK) {
      const float nn = fa * sn[tid] + ia * sk[tid];
      sn[tid] = nn;
      part = sq[tid] * round_to<T>(nn);
    }
    if (warp < (DK + 31) / 32) {
      part = warp_all_sum(part);
      if (lane == 0) s_red[warp] = part;
    }
    __syncthreads();
    float qn = 0.f;
#pragma unroll
    for (int w = 0; w < (DK + 31) / 32; ++w) qn += s_red[w];
    qn = round_to<T>(qn);
    const float denom = p.siging == 2 ? 1.f : fmaxf(fabsf(qn), expf(-m_new)) + p.eps;  // native_step.py:88-91
    if (rg == 0) hp[(int64_t)t * p.h_ss + j] = from_f32<T>(round_to<T>(acc) / denom);
    m = m_new;
  }
  if (p.c1) {
    float* dst = p.c1 + (int64_t)bh * DK * DV;
#pragma unroll
    for (int r = 0; r < RPT; ++r) dst[(int64_t)(rg + r * TPC) * DV + j] = C[r];
    __syncthreads();
    if (tid < DK) p.n1[(int64_t)bh * DK + tid] = sn[tid];
    if (tid == 0) p.m1[bh] = m;
  }
}

// (DHQK, DHHV) pairs with a k_recurrent instantiation
bool recurrent_pair_ok(int DK, int DV) {
  return (DK == DV && (DK == 32 || DK == 64 || DK == 128)) || (DK == 32 && DV == 64) || (DK == 64 && DV == 128);
}

template <typename T>
int launch(const StepParams& p, int DK, int DV, cudaStream_t st) {
  const int grid = p.B * p.NH;
  if (DK == DV) {
    switch (DK) {
      case 32: k_recurrent<T, 32, 32><<<grid, kStepThreads, 0, st>>>(p); break;
      case 64: k_recurrent<T, 64, 64><<<grid, kStepThreads, 0, st>>>(p); break;
      case 128: k_recurrent<T, 128, 128><<<grid, kStepThreads, 0, st>>>(p); break;
    }
  } else if (DK == 32) {
    k_recurrent<T, 32, 64><<<grid, kStepThreads, 0, st>>>(p);
  } else {
    k_recurrent<T, 64, 128><<<grid, kStepThreads, 0, st>>>(p);
  }
  count_launch();
  MLSTM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

int recurrent_sequence(const mlstm_b200_recurrent_args& a, cudaStream_t st) {
  if (!recurrent_pair_ok(a.DHQK, a.DHHV)) {
    set_error("recurrent kernels cover (DHQK, DHHV) = (32, 32), (64, 64), (128, 128), (32, 64) and (64, 128) (got %d, %d)",
              a.DHQK, a.DHHV);
    return MLSTM_B200_EUNSUPPORTED;
  }
  if (!a.q.ptr || !a.k.ptr || !a.v.ptr || !a.i.ptr || !a.f.ptr || !a.h.ptr) {
    set_error("q / k / v / i / f / h must not be NULL");
    return MLSTM_B200_EINVAL;
  }
  if (a.q.stride[3] != 1 || a.k.stride[3] != 1 || a.v.stride[3] != 1 || a.h.stride[3] != 1) {
    set_error("innermost stride of q / k / v / h must be 1");
    return MLSTM_B200_EINVAL;
  }
  const int ninit = (a.c_initial != 0) + (a.n_initial != 0) + (a.m_initial != 0);
  const int nlast = (a.c_last != 0) + (a.n_last != 0) + (a.m_last != 0);
  if ((ninit != 0 && ninit != 3) || (nlast != 0 && nlast != 3)) {
    set_error("initial / last states must be given all three or none");
    return MLSTM_B200_EINVAL;
  }
  if (a.B <= 0 || a.NH <= 0 || a.S <= 0) return 0;
  StepParams p{};
  p.B = a.B; p.NH = a.NH; p.S = a.S; p.siging = a.siging;
  p.eps = a.eps;
  p.scale = 1.f / sqrtf((float)a.DHQK);
  p.q = a.q.ptr; p.q_sb = a.q.stride[0]; p.q_sh = a.q.stride[1]; p.q_ss = a.q.stride[2];
  p.k = a.k.ptr; p.k_sb = a.k.stride[0]; p.k_sh = a.k.stride[1]; p.k_ss = a.k.stride[2];
  p.v = a.v.ptr; p.v_sb = a.v.stride[0]; p.v_sh = a.v.stride[1]; p.v_ss = a.v.stride[2];
  p.ig = a.i.ptr; p.i_sb = a.i.stride[0]; p.i_sh = a.i.stride[1]; p.i_ss = a.i.stride[2];
  p.fg = a.f.ptr; p.f_sb = a.f.stride[0]; p.f_sh = a.f.stride[1]; p.f_ss = a.f.stride[2];
  p.h = a.h.ptr; p.h_sb = a.h.stride[0]; p.h_sh = a.h.stride[1]; p.h_ss = a.h.stride[2];
  p.c0 = a.c_initial; p.n0 = a.n_initial; p.m0 = a.m_initial;
  p.c1 = a.c_last; p.n1 = a.n_last; p.m1 = a.m_last;
  MLSTM_DISPATCH_DTYPE(a.dtype, T, return launch<T>(p, a.DHQK, a.DHHV, st));
  return 0;
}

}  // namespace mlstm
