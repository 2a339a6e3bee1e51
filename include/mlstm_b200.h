/*
 * mlstm_b200.h -- C-ABI of the B200 (sm_100a) mLSTM chunkwise forward/backward.
 *
 * This is the drop-in boundary of the hot path.  The reference has no FFI of its
 * own (it is pure Python); the entry points below are what a binding for this
 * path replaces, one to one (paths relative to the reference root):
 *
 *   mlstm_b200_chunkwise_fw   <->  mlstm_chunkwise_fw
 *                                  mlstm_kernels/torch/chunkwise/native/fw.py:224-318
 *                                  (called from _mlstm_chunkwise_fwbw.forward,
 *                                   mlstm_kernels/torch/chunkwise/native/fwbw.py:36-102)
 *   mlstm_b200_chunkwise_bw   <->  mlstm_chunkwise_bw
 *                                  mlstm_kernels/torch/chunkwise/native/bw.py:206-348
 *                                  (called from _mlstm_chunkwise_fwbw.backward, fwbw.py:104-171)
 *
 * Conventions
 *   - plain C: device pointers, element strides, sizes; no torch types.
 *   - every call is asynchronous on the cudaStream_t passed in (as void*), holds no
 *     global mutable state besides a per-thread error string, and allocates no
 *     device memory: scratch is a caller-owned workspace whose size is returned by
 *     mlstm_b200_workspace_bytes().
 *   - return value: 0 on success, a negative MLSTM_B200_E* code for invalid
 *     arguments, a positive cudaError_t for CUDA failures.  Never exits / throws.
 *   - there is NO CPU fallback: on a machine without an sm_100 device every compute
 *     entry point returns an error.
 *
 * Tensor layout (same as the reference API, native/fwbw.py:228-243):
 *   q, k  (B, NH, S, DHQK)   v, h, dh (B, NH, S, DHHV)   i, f (B, NH, S)
 *   given as a base pointer plus ELEMENT strides in that index order; the innermost
 *   stride of q/k/v/dh must be 1 (the BSHD-strided views MatrixLSTMCell.forward
 *   creates, vision_lstm2.py:718-727, are consumed without a copy).
 *   States C (B, NH, DHQK, DHHV), n (B, NH, DHQK), m (B, NH) are contiguous fp32.
 */
#ifndef MLSTM_B200_H_
#define MLSTM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLSTM_B200_ABI_VERSION 4

/* element types of q/k/v/i/f/h and of the gradients */
enum { MLSTM_B200_F32 = 0, MLSTM_B200_BF16 = 1, MLSTM_B200_F16 = 2 };

/* error codes (negative); positive return values are cudaError_t */
enum {
  MLSTM_B200_OK = 0,
  MLSTM_B200_EINVAL = -1,      /* bad shape / stride / null pointer */
  MLSTM_B200_EUNSUPPORTED = -2,/* shape or dtype outside what the kernels cover */
  MLSTM_B200_EWORKSPACE = -3,  /* workspace too small */
  MLSTM_B200_ENODEVICE = -4    /* no sm_100 device / driver entry point missing */
};

/* kernel families; AUTO picks tensor-core (tcgen05) kernels for 16-bit inputs with
 * supported head dims and the exact fp32 FFMA kernels otherwise.  This selects between
 * precision modes of the SAME sm_100a path, not between backends. */
enum { MLSTM_B200_IMPL_AUTO = 0, MLSTM_B200_IMPL_EXACT = 1, MLSTM_B200_IMPL_TENSOR = 2 };

typedef struct mlstm_b200_tensor {
  void* ptr;         /* device pointer (may be NULL for optional tensors) */
  int64_t stride[4]; /* element strides, index order as documented above; unused = 0 */
} mlstm_b200_tensor;

typedef struct mlstm_b200_shape {
  int32_t B, NH, S, DHQK, DHHV;
  int32_t chunk_size; /* S % chunk_size == 0 is required (native/fw.py:252-254) */
  int32_t dtype;      /* MLSTM_B200_F32 / BF16 / F16 */
  int32_t impl;       /* MLSTM_B200_IMPL_* */
  int32_t reverse;    /* 1: anti-causal scan, h = flip(mLSTM(flip(inputs))) along S without any copy
                         (the ROWWISE_FROM_BOT_RIGHT direction of ViLLayer, vision_lstm2.py:292-312);
                         initial / last states then refer to the END / START of the sequence in memory */
  int32_t siging;     /* 1: sigmoid input gate, no max state, denominator max(|n|, 1) -- the variant the
                         reference's CUDA model path uses (triton_xl_chunk_siging/fwbw.py:211-268,
                         parallel/native_siging/fw.py:15-74); m_initial / m_last are then ignored / zero.
                         2: the same sigmoid input gate WITHOUT the normaliser (the reference's normalize=False,
                         triton_xl_chunk_siging/fwbw.py:211-268): h = q C + sum_s P_ts v_s is the numerator, eps does not
                         enter it, and the backward uses dh as it is and never reads n_out (the forward still writes
                         n_out / m_out and carries n, so the last states are those of siging = 1).  Not with the fused
                         cell-output epilogue (MLSTM_B200_EUNSUPPORTED).  Any other value: MLSTM_B200_EINVAL. */
  float eps;
  float qk_scale;     /* <= 0 selects DHQK^-0.5 (native/fw.py:263-264) */
  float gate_soft_cap;/* > 0: i and f are gate PRE-activations and the kernels apply the cell's soft cap
                         cap * tanh(x / cap) themselves (MatrixLSTMCell.soft_cap, vision_lstm2.py:714-715, 755-756)
                         while scanning; di / df are then gradients w.r.t. the pre-activations (the factor
                         1 - tanh^2(x / cap) is applied at the store).  Tensor-core route only: the exact route
                         returns MLSTM_B200_EUNSUPPORTED for gate_soft_cap > 0.  <= 0: i / f are used as given. */
  int32_t grad_dtype; /* backward only: dtype of dq / dk / dv / di / df.  0 = shape.dtype.  MLSTM_B200_F16 with a BF16 kernel
                         (or the reverse) writes the gradients in the CALLER's 16-bit dtype straight from the fp32
                         accumulators -- a bf16 kernel under fp16 autocast (native/fwbw.py:37 casts the inputs, autograd casts
                         the gradients back) then needs no cast pass over dq / dk / dv.  Tensor-core route only. */
} mlstm_b200_shape;

/* Optional fused cell-output epilogue of the forward (SURVEY.md section 8(f) #3): instead of (or in addition to) h the
 * kernel writes
 *     y[b,hd,s,d] = (h - mean) * rstd * weight[c] + bias[c] + skip[c] * x[b,hd,s,d],   c = hd * DHHV + d
 * with mean / rstd over the DHHV elements of one (token, head) row of h rounded to the kernel dtype (biased variance,
 * rstd = (var + eps)^-1/2) -- MultiHeadLayerNorm (vision_lstm2.py:928-944) on the cell's output, ViLLayer's learnable
 * skip (vision_lstm2.py:306) and, through y's strides, the (B, NH, S, D) -> (B, S, NH*D) relayout (vision_lstm2.py:749-751)
 * -- from the registers that hold the row in the epilogue anyway: in inference h never reaches HBM un-normalised; in
 * training h is still written (fw_args.h) because the LayerNorm backward needs it (mlstm_b200_cellout_bw).
 * y and x are (B, NH, S, DHHV) views given by element strides, innermost stride 1, 16-byte aligned with strides that are
 * multiples of 8 elements (y goes out through a TMA tensor map); both are 16-bit, of dtype xy_dtype (BF16 or F16), which
 * may differ from shape.dtype (bf16 kernel under fp16 autocast).  weight / bias / skip: contiguous fp32 (NH*DHHV), each
 * may be NULL (1 / 0 / 0); x.ptr may be NULL.  Tensor-core route only, every head geometry it covers: DHQK == DHHV and
 * the rectangular (DHQK, DHHV) = (32, 64), (64, 128), whose two DHQK-wide column blocks per head run as one two-CTA
 * cluster that exchanges the row statistics (mean and rstd are those of the whole DHHV row). */
typedef struct mlstm_b200_fw_epilogue {
  mlstm_b200_tensor y; /* out */
  mlstm_b200_tensor x; /* optional skip input */
  const float* weight;
  const float* bias;
  const float* skip;
  float eps;
  int32_t xy_dtype;
} mlstm_b200_fw_epilogue;

typedef struct mlstm_b200_fw_args {
  mlstm_b200_shape shape;
  /* inputs */
  mlstm_b200_tensor q, k, v, i, f;
  const float* c_initial; /* optional, all three or none */
  const float* n_initial;
  const float* m_initial;
  /* outputs */
  mlstm_b200_tensor h;    /* dtype, strides given (contiguous BHSD is the usual case) */
  float* n_out;           /* (B, NH, S) fp32: max(|den|, exp(-m)) saved for backward */
  float* m_out;           /* (B, NH, S) fp32: per-token stabiliser saved for backward */
  float* c_last;          /* optional last states, all three or none */
  float* n_last;
  float* m_last;
  void* c_states;         /* optional: per-tile C states for the backward, mlstm_b200_states_bytes()
                             bytes (the reference's return_all_states mode, native/fwbw.py:73-101) */
  void* workspace;
  size_t workspace_bytes;
  const mlstm_b200_fw_epilogue* epilogue; /* optional; with it h.ptr may be NULL (no un-normalised h is written) */
} mlstm_b200_fw_args;

typedef struct mlstm_b200_bw_args {
  mlstm_b200_shape shape;
  /* forward inputs and saved vectors */
  mlstm_b200_tensor q, k, v, i, f;
  const float* c_initial;
  const float* n_initial;
  const float* m_initial;
  const float* n_out;
  const float* m_out;
  const void* c_states;   /* optional: what the forward wrote; NULL = recompute (native/bw.py:251-266) */
  /* incoming gradients */
  mlstm_b200_tensor dh;
  const float* dc_last;   /* optional (B, NH, DHQK, DHHV) */
  /* outputs */
  mlstm_b200_tensor dq, dk, dv; /* dtype */
  mlstm_b200_tensor di, df;     /* dtype, (B, NH, S) */
  float* dc_initial;            /* optional; written iff non-NULL */
  void* workspace;
  size_t workspace_bytes;
} mlstm_b200_bw_args;

/* ABI version of the loaded library (== MLSTM_B200_ABI_VERSION it was built with). */
int mlstm_b200_abi_version(void);

/* Human-readable description of the last error on the calling thread ("" if none). */
const char* mlstm_b200_last_error(void);

/* Bytes of scratch the forward (backward = 0) or backward (backward = 1) needs. */
size_t mlstm_b200_workspace_bytes(const mlstm_b200_shape* shape, int backward);

/* Bytes of the optional c_states buffer (0 when the selected kernels recompute the states). */
size_t mlstm_b200_states_bytes(const mlstm_b200_shape* shape);

/* 1 if the tensor-core (tcgen05) kernels cover this shape/dtype forward AND backward, else 0
 * (16-bit dtypes, S % 4 == 0, and DHQK == DHHV in {32, 64, 128} or (DHQK, DHHV) in {(32, 64), (64, 128)}; the
 * head-dim-128 backward runs as four head-dim-64 block problems inside the call, a rectangular (D, 2 D) call as two
 * square head-dim-D problems on the two column halves of v / h / dh / dv).  The forward's fused cell-output epilogue
 * (mlstm_b200_fw_epilogue) is available for every shape this returns 1 for. */
int mlstm_b200_tensor_path_supported(const mlstm_b200_shape* shape);

/* Forward: h, n_out, m_out and optionally the last (C, n, m) states. */
int mlstm_b200_chunkwise_fw(const mlstm_b200_fw_args* args, void* cuda_stream);

/* Backward (n_out and all max states are constants, native/bw.py:44-47):
 * dq, dk, dv, di, df and optionally dC_initial. */
int mlstm_b200_chunkwise_bw(const mlstm_b200_bw_args* args, void* cuda_stream);

/* Number of kernels the last fw / bw call on this thread launched (for bench.py's
 * gpu_launches claim). */
int mlstm_b200_last_launch_count(void);

/* Profiling hook of the PROFILE build (lib/libmlstm_b200_prof.so, compiled with -DMLSTM_TC_PROFILE): when set to
 * a device buffer of at least 8192 int64, CTA 0 of the tensor-core kernels records clock64() at its phase
 * boundaries (forward at [tile*16 + slot], backward at [4096 + tile*16 + slot]).  NULL disables it.
 * In the product library this is a no-op: the product build holds no process-global mutable state. */
void mlstm_b200_debug_set_clock_buffer(void* dev_ptr);

/* How many {2, 1, 1} clusters of the forward with the fused epilogue for rectangular heads (shape.DHQK != DHHV; see
 * mlstm_b200_fw_epilogue) the current device can hold at once (cudaOccupancyMaxActiveClusters); 0 for a shape that does
 * not launch as clusters, -1 on error. */
int mlstm_b200_debug_fw_epilogue_clusters(const mlstm_b200_shape* shape);

/* ---------------------------------------------------------------------------------------------
 * Recurrent form (SURVEY.md section 8(f) #4): S token-by-token steps of the mLSTM with the (C, n, m) state kept on
 * chip for the whole call.  S = 1 is the step kernel
 *   mlstm_recurrent_step__native_fw      mlstm_kernels/torch/recurrent/native_step.py:8-101
 * and S > 1 the sequence loop around it
 *   _mlstm_recurrent_sequence_loop_fw    mlstm_kernels/torch/recurrent/native_sequence.py:14-130
 * which the reference's inference wrapper runs for the tokens that do not fill a chunk
 * (wrap_chunkwise__arbitrary_sequence_length, mlstm_kernels/torch/kernel_wrappers.py:12-201).
 *   q, k (B, NH, S, DHQK), v, h (B, NH, S, DHHV), i, f (B, NH, S): element strides [b, head, s, 1] / [b, head, s];
 *   DHQK == DHHV in {32, 64, 128} or (DHQK, DHHV) in {(32, 64), (64, 128)}; dtype of q / k / v / i / f / h; states
 *   contiguous fp32 as in the chunkwise calls
 *   (m is (B, NH)).  Initial states: all three or none (none = zeros); last states: all three or none; the last
 *   states may alias the initial ones (in-place update).  siging = 1: sigmoid input gate, m stays 0; siging = 2: the
 *   same without the normaliser (h = q . C_t, as mlstm_b200_shape::siging = 2).
 *   Forward only (the reference's recurrent kernels have no backward).
 */
typedef struct mlstm_b200_recurrent_args {
  int32_t B, NH, S, DHQK, DHHV;
  int32_t dtype;  /* MLSTM_B200_F32 / BF16 / F16 */
  int32_t siging;
  float eps;
  mlstm_b200_tensor q, k, v, i, f;
  const float* c_initial;
  const float* n_initial;
  const float* m_initial;
  mlstm_b200_tensor h; /* out */
  float* c_last;
  float* n_last;
  float* m_last;
} mlstm_b200_recurrent_args;

int mlstm_b200_recurrent_sequence(const mlstm_b200_recurrent_args* args, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------
 * The cell's output stage (SURVEY.md section 8(f) #3: the callers either side of the path).
 *
 *   y[b,s,hd*D+d] = (h[b,hd,s,d] - mean) * rstd * weight[c] + bias[c] + skip[c] * x[b,s,c]
 *
 * with mean / rstd over the D elements of one (token, head) group (biased variance, rstd = (var+eps)^-1/2).
 * One pass replaces, in the reference:
 *   MultiHeadLayerNorm.forward       ultralytics/nn/modules/vision_lstm/vision_lstm2.py:928-944
 *   MatrixLSTMCell.forward tail      vision_lstm2.py:749-751 (h.to(dtype), transpose + reshape copy)
 *   ViLLayer.mlstm_branch skip add   vision_lstm2.py:306     (h + learnable_skip * x_qk_conv_act)
 * and mlstm_b200_cellout_bw replaces their autograd backward.
 *   h, dh   (B, NH, S, D)  element strides [b, head, s, 1], h_dtype
 *   x, y, dy, dx (B, S, NH*D)  element strides [b, s, 1];  x and y share one dtype (x_dtype == y_dtype)
 *   weight (= 1 + MultiHeadLayerNorm.weight, the reference's weight_proxy, vision_lstm2.py:900-907),
 *   bias, skip: contiguous fp32 (NH*D); weight / bias may be NULL (1 / 0); x.ptr == NULL drops the skip term.
 * Supported: D in {32, 64, 128}, NH*D a multiple of 128 and <= 2048; pointers 8-byte (16-bit types) or
 * 16-byte (fp32) aligned, strides multiples of 4 elements; x has y's strides; in the backward dh has h's strides
 * and x / dx have dy's (the kernels walk each family with one running offset).
 */
typedef struct mlstm_b200_cellout_args {
  int32_t B, NH, S, D;
  int32_t h_dtype, x_dtype, y_dtype; /* MLSTM_B200_F32 / BF16 / F16 */
  float eps;
  mlstm_b200_tensor h;
  mlstm_b200_tensor x; /* optional */
  mlstm_b200_tensor y; /* out */
  const float* weight;
  const float* bias;
  const float* skip;
} mlstm_b200_cellout_args;

typedef struct mlstm_b200_cellout_bw_args {
  mlstm_b200_cellout_args fw; /* h, x, weight, skip as given to the forward (y is ignored) */
  mlstm_b200_tensor dy;       /* incoming gradient, y_dtype */
  mlstm_b200_tensor dh;       /* out, h_dtype */
  mlstm_b200_tensor dx;       /* out, x_dtype: dy * skip; optional */
  float* dweight;             /* out (NH*D) fp32, each optional */
  float* dbias;
  float* dskip;
  void* workspace;            /* mlstm_b200_cellout_workspace_bytes() bytes (CTA partial sums) */
  size_t workspace_bytes;
} mlstm_b200_cellout_bw_args;

size_t mlstm_b200_cellout_workspace_bytes(const mlstm_b200_cellout_args* args);
int mlstm_b200_cellout_fw(const mlstm_b200_cellout_args* args, void* cuda_stream);
int mlstm_b200_cellout_bw(const mlstm_b200_cellout_bw_args* args, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------
 * RMSNorm in front of the branch: ViLLayer.norm / .ffn_norm = nn.RMSNorm(dim, eps=1e-6, elementwise_affine)
 * (vision_lstm2.py:277-278, applied at :318-327).  y = round_x(x * rsqrt(mean(x^2) + eps)) * weight over the last
 * dimension of a dense (rows, C) matrix -- the rounding of the normalised row to the input dtype is what torch's
 * composite rms_norm does when input and weight dtypes differ (fp16 autocast).  rstd (rows) fp32 is written by the
 * forward and read by the backward.  C in {192, 256, 384, 512}; x / dx of x_dtype, y / dy of y_dtype.
 */
typedef struct mlstm_b200_rmsnorm_args {
  int64_t rows;
  int32_t C;
  int32_t x_dtype, y_dtype;
  float eps;
  const void* x;
  void* y;             /* out (forward) */
  const float* weight; /* (C) fp32 or NULL (= 1) */
  float* rstd;         /* (rows) fp32: out (forward), in (backward) */
} mlstm_b200_rmsnorm_args;

typedef struct mlstm_b200_rmsnorm_bw_args {
  mlstm_b200_rmsnorm_args fw; /* x, weight, rstd as in the forward (y is ignored) */
  const void* dy;
  void* dx;                   /* out, x_dtype */
  float* dweight;             /* out (C) fp32, optional */
  void* workspace;            /* mlstm_b200_rmsnorm_workspace_bytes() bytes */
  size_t workspace_bytes;
} mlstm_b200_rmsnorm_bw_args;

size_t mlstm_b200_rmsnorm_workspace_bytes(const mlstm_b200_rmsnorm_args* args);
int mlstm_b200_rmsnorm_fw(const mlstm_b200_rmsnorm_args* args, void* cuda_stream);
int mlstm_b200_rmsnorm_bw(const mlstm_b200_rmsnorm_bw_args* args, void* cuda_stream);

/* Re-round a contiguous buffer of n 16-bit elements fp16 -> bf16 or bf16 -> fp16 (one RN rounding through fp32,
 * bit-identical to Tensor.to()): the cast the reference's kernels apply to q / k / v under CUDA autocast
 * (custom_fwd(cast_inputs=autocast_kernel_dtype), native/fwbw.py:37) as one streaming pass at HBM rate.  src and dst
 * may not overlap unless identical (in place). */
int mlstm_b200_convert16(const void* src, void* dst, int64_t n, int32_t src_dtype, int32_t dst_dtype, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* MLSTM_B200_H_ */
