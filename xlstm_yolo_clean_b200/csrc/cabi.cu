// extern "C" entry points declared in include/mlstm_b200.h: argument validation and
// dispatch to the exact (fp32 FFMA) or tensor-core (tcgen05) kernel family.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"

namespace mlstm {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches += n; }

namespace {

int check_qkv(const mlstm_b200_tensor& t, const char* name) {
  if (!t.ptr) {
    set_error("%s is NULL", name);
    return MLSTM_B200_EINVAL;
  }
  if (t.stride[3] != 1) {
    set_error("%s: innermost stride must be 1 (got %lld)", name, (long long)t.stride[3]);
    return MLSTM_B200_EINVAL;
  }
  return 0;
}
int check_vec(const mlstm_b200_tensor& t, const char* name) {
  if (!t.ptr) {
    set_error("%s is NULL", name);
    return MLSTM_B200_EINVAL;
  }
  return 0;
}

int check_siging(int32_t siging) {
  if (siging < 0 || siging > 2) {
    set_error("siging must be 0, 1 or 2 (got %d)", siging);
    return MLSTM_B200_EINVAL;
  }
  return 0;
}

int require_device() {
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    set_error("no CUDA device: %s", cudaGetErrorString(e));
    return MLSTM_B200_ENODEVICE;
  }
  // The tensor maps are encoded through the DRIVER API, which needs the device's primary context bound to the
  // calling thread.  A fresh thread -- e.g. PyTorch's autograd thread running the first backward of a process,
  // with its allocations served from the caching allocator -- may not have made a runtime call that binds it yet.
  // (cudaFree(0) binds it; it is only issued when no context is current, so never inside a stream capture.)
  static thread_local int bound_dev = -1;
  if (bound_dev != dev) {
    if (!tensor_context_is_current()) {
      e = cudaFree(0);
      if (e != cudaSuccess) {
        set_error("cannot bind the CUDA context of device %d: %s", dev, cudaGetErrorString(e));
        return MLSTM_B200_ENODEVICE;
      }
    }
    bound_dev = dev;
  }
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) {
    set_error("device %d has compute capability %d.x; this library is built for sm_100a only", dev, major);
    return MLSTM_B200_ENODEVICE;
  }
  return 0;
}

bool use_tensor(const mlstm_b200_shape& s, int* err) {
  *err = 0;
  if (s.impl == MLSTM_B200_IMPL_EXACT) return false;
  bool ok = tensor_supported(s);
  if (s.impl == MLSTM_B200_IMPL_TENSOR && !ok) {
    set_error("tensor-core path does not cover dtype=%d DHQK=%d DHHV=%d chunk=%d", s.dtype, s.DHQK, s.DHHV,
              s.chunk_size);
    *err = MLSTM_B200_EUNSUPPORTED;
  }
  return ok;
}

// Validation and route choice of mlstm_b200_chunkwise_fw (Args = mlstm_b200_fw_args) and _bw (mlstm_b200_bw_args), in
// the order the checks run; *tc: the call goes to the tensor-core kernels, otherwise to the exact ones.
template <typename Args>
int chunkwise_route(const Args& a, bool* tc) {
  constexpr bool bw = std::is_same<Args, mlstm_b200_bw_args>::value;
  const mlstm_b200_shape& s = a.shape;
  if (int e = check_qkv(a.q, "q")) return e;
  if (int e = check_qkv(a.k, "k")) return e;
  if (int e = check_qkv(a.v, "v")) return e;
  if constexpr (bw) {
    if (int e = check_qkv(a.dh, "dh")) return e;
    if (int e = check_qkv(a.dq, "dq")) return e;
    if (int e = check_qkv(a.dk, "dk")) return e;
    if (int e = check_qkv(a.dv, "dv")) return e;
  } else if (a.epilogue) {  // fused cell-output epilogue: y is mandatory, the un-normalised h optional
    if (int e = check_qkv(a.epilogue->y, "epilogue.y")) return e;
    if (a.h.ptr)
      if (int e = check_qkv(a.h, "h")) return e;
  } else if (int e = check_qkv(a.h, "h")) {
    return e;
  }
  if (int e = check_vec(a.i, "i")) return e;
  if (int e = check_vec(a.f, "f")) return e;
  if constexpr (bw) {
    if (int e = check_vec(a.di, "di")) return e;
    if (int e = check_vec(a.df, "df")) return e;
  }
  if (!a.n_out || !a.m_out) {
    set_error("n_out / m_out are NULL");
    return MLSTM_B200_EINVAL;
  }
  int ninit = (a.c_initial != 0) + (a.n_initial != 0) + (a.m_initial != 0);
  if constexpr (bw) {
    if (ninit != 0 && ninit != 3) {
      set_error("initial states must be given all three or none");
      return MLSTM_B200_EINVAL;
    }
  } else {
    int nlast = (a.c_last != 0) + (a.n_last != 0) + (a.m_last != 0);
    if ((ninit != 0 && ninit != 3) || (nlast != 0 && nlast != 3)) {
      set_error("initial / last states must be given all three or none");
      return MLSTM_B200_EINVAL;
    }
  }
  if (s.S % (s.chunk_size > 0 ? s.chunk_size : 1)) {
    set_error("Sequence length %d is not divisible by chunk size %d.", s.S, s.chunk_size);
    return MLSTM_B200_EINVAL;
  }
  if (int e = check_siging(s.siging)) return e;
  if constexpr (!bw) {
    if (a.epilogue && s.siging == 2) {  // the cell it fuses (MatrixLSTMCell) always normalises
      set_error("the fused cell-output epilogue does not cover siging = 2 (no normaliser)");
      return MLSTM_B200_EUNSUPPORTED;
    }
  }
  if (int e = require_device()) return e;
  int err = 0;
  *tc = use_tensor(s, &err);
  if (err) return err;
  // AUTO accepts any strides like the reference does (torch/utils.py:30-42): views a TMA tensor map cannot describe
  // (odd offsets, strides that are not multiples of 16 bytes) go to the exact kernels, which take any stride.  The
  // exact family needs its own (larger) workspace: mlstm_b200_workspace_bytes with impl = EXACT.
  if (*tc && s.impl == MLSTM_B200_IMPL_AUTO && !tensor_views_ok(a)) *tc = false;
  if (!*tc && s.gate_soft_cap > 0.f) {
    set_error("gate_soft_cap is applied by the tensor-core kernels only; cap the gates before an exact-route call");
    return MLSTM_B200_EUNSUPPORTED;
  }
  if constexpr (bw) {
    const int gd = s.grad_dtype;
    if (gd != 0 && gd != s.dtype) {
      if (gd != MLSTM_B200_BF16 && gd != MLSTM_B200_F16) {
        set_error("grad_dtype must be 0, MLSTM_B200_BF16 or MLSTM_B200_F16 (got %d)", gd);
        return MLSTM_B200_EINVAL;
      }
      if (!*tc) {
        set_error("gradients in a dtype other than shape.dtype are written by the tensor-core kernels only");
        return MLSTM_B200_EUNSUPPORTED;
      }
    }
  } else if (!*tc && a.epilogue) {
    set_error("the fused cell-output epilogue exists on the tensor-core route only (use mlstm_b200_cellout_fw)");
    return MLSTM_B200_EUNSUPPORTED;
  }
  return 0;
}

}  // namespace
}  // namespace mlstm

using namespace mlstm;

extern "C" {

int mlstm_b200_abi_version(void) { return MLSTM_B200_ABI_VERSION; }

const char* mlstm_b200_last_error(void) { return g_err; }

int mlstm_b200_last_launch_count(void) { return g_launches; }

void mlstm_b200_debug_set_clock_buffer(void* dev_ptr) { tensor_set_clock_buffer(dev_ptr); }

int mlstm_b200_debug_fw_epilogue_clusters(const mlstm_b200_shape* shape) {
  g_err[0] = 0;
  if (!shape) {
    set_error("shape is NULL");
    return -1;
  }
  if (require_device()) return -1;
  return tensor_fw_epilogue_clusters(*shape);
}

int mlstm_b200_tensor_path_supported(const mlstm_b200_shape* shape) {
  if (!shape) return 0;
  return tensor_supported(*shape) ? 1 : 0;
}

size_t mlstm_b200_states_bytes(const mlstm_b200_shape* shape) {
  if (!shape) return 0;
  int err = 0;
  return use_tensor(*shape, &err) ? tensor_states_bytes(*shape) : 0;
}

size_t mlstm_b200_workspace_bytes(const mlstm_b200_shape* shape, int backward) {
  if (!shape) return 0;
  int err = 0;
  size_t n = use_tensor(*shape, &err) ? tensor_workspace_bytes(*shape, backward)
                                      : exact_workspace_bytes(*shape, backward);
  return n < 256 ? 256 : n;
}

int mlstm_b200_chunkwise_fw(const mlstm_b200_fw_args* a, void* stream) {
  g_err[0] = 0;
  g_launches = 0;
  if (!a) {
    set_error("args is NULL");
    return MLSTM_B200_EINVAL;
  }
  bool tc = false;
  if (int e = chunkwise_route(*a, &tc)) return e;
  return tc ? tensor_fw(*a, (cudaStream_t)stream) : exact_fw(*a, (cudaStream_t)stream);
}

int mlstm_b200_chunkwise_bw(const mlstm_b200_bw_args* a, void* stream) {
  g_err[0] = 0;
  g_launches = 0;
  if (!a) {
    set_error("args is NULL");
    return MLSTM_B200_EINVAL;
  }
  bool tc = false;
  if (int e = chunkwise_route(*a, &tc)) return e;
  return tc ? tensor_bw(*a, (cudaStream_t)stream) : exact_bw(*a, (cudaStream_t)stream);
}

int mlstm_b200_recurrent_sequence(const mlstm_b200_recurrent_args* a, void* stream) {
  g_err[0] = 0;
  g_launches = 0;
  if (!a) {
    set_error("args is NULL");
    return MLSTM_B200_EINVAL;
  }
  if (int e = check_siging(a->siging)) return e;
  if (int e = require_device()) return e;
  return recurrent_sequence(*a, (cudaStream_t)stream);
}

size_t mlstm_b200_cellout_workspace_bytes(const mlstm_b200_cellout_args* a) {
  if (!a) return 0;
  size_t n = cellout_workspace_bytes(*a);
  return n < 256 ? 256 : n;
}

int mlstm_b200_cellout_fw(const mlstm_b200_cellout_args* a, void* stream) {
  g_err[0] = 0;
  g_launches = 0;
  if (!a) {
    set_error("args is NULL");
    return MLSTM_B200_EINVAL;
  }
  if (int e = require_device()) return e;
  return cellout_fw(*a, (cudaStream_t)stream);
}

int mlstm_b200_cellout_bw(const mlstm_b200_cellout_bw_args* a, void* stream) {
  g_err[0] = 0;
  g_launches = 0;
  if (!a) {
    set_error("args is NULL");
    return MLSTM_B200_EINVAL;
  }
  if (int e = require_device()) return e;
  return cellout_bw(*a, (cudaStream_t)stream);
}

size_t mlstm_b200_rmsnorm_workspace_bytes(const mlstm_b200_rmsnorm_args* a) {
  if (!a) return 0;
  size_t n = rmsnorm_workspace_bytes(*a);
  return n < 256 ? 256 : n;
}

int mlstm_b200_rmsnorm_fw(const mlstm_b200_rmsnorm_args* a, void* stream) {
  g_err[0] = 0;
  g_launches = 0;
  if (!a) {
    set_error("args is NULL");
    return MLSTM_B200_EINVAL;
  }
  if (int e = require_device()) return e;
  return rmsnorm_fw(*a, (cudaStream_t)stream);
}

int mlstm_b200_rmsnorm_bw(const mlstm_b200_rmsnorm_bw_args* a, void* stream) {
  g_err[0] = 0;
  g_launches = 0;
  if (!a) {
    set_error("args is NULL");
    return MLSTM_B200_EINVAL;
  }
  if (int e = require_device()) return e;
  return rmsnorm_bw(*a, (cudaStream_t)stream);
}

int mlstm_b200_convert16(const void* src, void* dst, int64_t n, int32_t src_dtype, int32_t dst_dtype, void* stream) {
  g_err[0] = 0;
  g_launches = 0;
  if (int e = require_device()) return e;
  return convert16(src, dst, n, src_dtype, dst_dtype, (cudaStream_t)stream);
}

}  // extern "C"
