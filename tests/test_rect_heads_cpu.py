"""Support matrix of the tensor-core route for rectangular heads (DHQK != DHHV), read through
mlstm_b200_tensor_path_supported, which needs no device: 16-bit (32, 64) and (64, 128) are covered, every square
answer is what it was, and every other rectangular pair and fp32 stay on the exact route."""
import ctypes

import pytest

import __graft_entry__ as G


@pytest.fixture(scope="module")
def lib():
    G.build()
    import xlstm_yolo_clean_b200 as pkg

    return pkg.load_library()


def _supported(lib, DK, DV, dtype, S=256):
    from xlstm_yolo_clean_b200 import _cabi

    s = _cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype = 2, 4, S, DK, DV, 64, dtype
    return bool(lib.mlstm_b200_tensor_path_supported(ctypes.byref(s)))


def test_square_answers_unchanged(lib):
    from xlstm_yolo_clean_b200 import _cabi

    for D in (16, 32, 48, 64, 96, 128, 256):
        for dt in (_cabi.BF16, _cabi.F16):
            assert _supported(lib, D, D, dt) == (D in (32, 64, 128)), (D, dt)
        assert not _supported(lib, D, D, _cabi.F32)
    assert not _supported(lib, 64, 64, _cabi.BF16, S=198)  # S % 4 != 0


@pytest.mark.parametrize("DK,DV", [(32, 64), (64, 128)])
def test_rectangular_pairs_supported_in_16_bit(lib, DK, DV):
    from xlstm_yolo_clean_b200 import _cabi

    assert _supported(lib, DK, DV, _cabi.BF16) and _supported(lib, DK, DV, _cabi.F16)
    assert _supported(lib, DK, DV, _cabi.BF16, S=196)  # ragged last tile
    assert not _supported(lib, DK, DV, _cabi.F32)
    assert not _supported(lib, DK, DV, _cabi.BF16, S=198)


@pytest.mark.parametrize("DK,DV", [(16, 32), (64, 32), (128, 64), (128, 256), (32, 128), (64, 96)])
def test_other_rectangular_pairs_stay_on_the_exact_route(lib, DK, DV):
    from xlstm_yolo_clean_b200 import _cabi

    for dt in (_cabi.BF16, _cabi.F16, _cabi.F32):
        assert not _supported(lib, DK, DV, dt)


def test_rectangular_state_and_workspace_sizes(lib):
    """c_states holds DHQK x DHHV 16-bit values per 128-token tile; the backward's workspace covers the block problems."""
    from xlstm_yolo_clean_b200 import _cabi

    for DK, DV in ((32, 64), (64, 128)):
        s = _cabi.Shape()
        s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype, s.impl = 2, 3, 196, DK, DV, 4, _cabi.BF16, _cabi.IMPL_AUTO
        assert lib.mlstm_b200_states_bytes(ctypes.byref(s)) == 2 * 3 * 2 * DK * DV * 2
        assert lib.mlstm_b200_workspace_bytes(ctypes.byref(s), 1) > 0
