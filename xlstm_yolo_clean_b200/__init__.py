"""B200-native (sm_100a) mLSTM chunkwise forward/backward behind the mlstm_kernels interface.

Public API (mirrors mlstm_kernels/torch/chunkwise/native/fwbw.py:228-263 and the registry in
mlstm_kernels/torch/chunkwise/__init__.py:9-15 of the reference):

    mlstm_chunkwise__b200(q, k, v, i, f, c_initial=None, n_initial=None, m_initial=None,
                          return_last_states=False, eps=1e-6, chunk_size=64,
                          autocast_kernel_dtype=torch.bfloat16, **kwargs)
    register()            add "chunkwise--b200" to the reference registry (if importable)
    patch_model(model)    point every MatrixLSTMCell.gpu_backend at the new kernel; ``fused=True`` also
                          rebinds ViLLayer.mlstm_branch to the flip-free branch with the fused cell output
    cell_out(h, ...)      fused MultiHeadLayerNorm + relayout + learnable skip (vision_lstm2.py:928-944, 306)
"""
from ._cabi import LIB_PATH, LibraryMissing, load_library  # noqa: F401
from .host_pipeline import HostFwBw  # noqa: F401
from .vil import (cell_out, cellout_supported, mlstm_branch_b200, mlstm_cell_b200, patch_layers, rms_norm_b200,  # noqa: F401
                  rmsnorm_supported)
from .backend import (  # noqa: F401
    KERNEL_NAME,
    last_launch_count,
    mlstm_chunkwise__b200,
    mlstm_chunkwise_bw,
    mlstm_chunkwise_fw,
    mlstm_recurrent_sequence__b200,
    mlstm_recurrent_step__b200,
    convert16,
    mlstm_siging_chunkwise__b200,
    patch_model,
    register,
    set_default_impl,
    tensor_path_supported,
)
