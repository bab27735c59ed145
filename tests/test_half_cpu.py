"""CPU: argument checks of the half-precision RoIAlign entry points (they run before any CUDA call) and of the Python
surface that feeds them."""
import ctypes

import pytest
import torch


def _err():
    from nuhtc_b200 import _lib as L
    return L.lib().nuhtc_last_error().decode()


def test_to_cg32_dt_rejects_bad_dtype_and_misaligned_pointers():
    from nuhtc_b200 import _lib as L
    lib = L.lib()
    ok_in, ok_out = 0x10000, 0x20000        # never dereferenced: the checks fail first
    assert lib.nuhtc_to_cg32_dt(ok_in, 3, ok_out, 1, 32, 4, 4, 0, None) == -1
    assert "unknown dtype code 3" in _err()
    assert lib.nuhtc_to_cg32_dt(ok_in, -1, ok_out, 1, 32, 4, 4, 0, None) == -1
    assert "unknown dtype code -1" in _err()
    # four input elements are read at a time: 8-byte alignment for 16-bit types, 16 bytes for fp32
    for code, bad in ((L.DTYPE_F16, ok_in + 2), (L.DTYPE_BF16, ok_in + 4), (L.DTYPE_F32, ok_in + 8)):
        assert lib.nuhtc_to_cg32_dt(bad, code, ok_out, 1, 32, 4, 4, 0, None) == -1
        assert "misaligned" in _err()
    assert lib.nuhtc_to_cg32_dt(ok_in, L.DTYPE_F16, ok_out + 8, 1, 32, 4, 4, 0, None) == -1
    assert "misaligned" in _err()
    # the fp32 entry point is the F32 case of the same checks
    assert lib.nuhtc_to_cg32(ok_in + 8, ok_out, 1, 32, 4, 4, 0, None) == -1
    assert "misaligned" in _err()


def _cg32_dt(out_ptr, code, K=1):
    from nuhtc_b200 import _lib as L
    Hs, Ws = (ctypes.c_int * 1)(8), (ctypes.c_int * 1)(8)
    sc = (ctypes.c_float * 1)(0.25)
    feats = (ctypes.c_void_p * 1)(0x40000)
    return L.lib().nuhtc_roi_align_cg32_dt(feats, Hs, Ws, sc, 1, 1, 32, 0x50000, K, 7, 7, 0, 1, L.ROI_ROUTE, 56.0, None, out_ptr,
                                           code, None, 0x60000, 1 << 20, None)


def test_roi_align_cg32_dt_rejects_bad_dtype_and_misaligned_out():
    from nuhtc_b200 import _lib as L
    assert _cg32_dt(0x70000, 7) == -1
    assert "unknown dtype code 7" in _err()
    assert _cg32_dt(0x70000, 7, K=0) == -1            # checked even when there is nothing to do
    for code in (L.DTYPE_F32, L.DTYPE_F16, L.DTYPE_BF16):
        for off in (2, 8):                              # bulk stores need 16-byte aligned outputs whatever the type
            assert _cg32_dt(0x70000 + off, code) == -1
            assert "out must be 16-byte aligned" in _err()


def test_mixed_dtype_levels_raise_value_error():
    import nuhtc_b200 as nb
    lv = [torch.zeros(1, 32, 8, 8, dtype=torch.float16), torch.zeros(1, 32, 4, 4, dtype=torch.float32)]
    with pytest.raises(ValueError, match="one dtype"):
        nb.roi_align_levels(lv, torch.zeros(1, 5), 7, [0.25, 0.125], 0)
    with pytest.raises(ValueError, match="one dtype"):
        nb.roi_align_levels([lv[0], lv[0].bfloat16()], torch.zeros(1, 5), 7, [0.25, 0.125], 0)
    with pytest.raises(ValueError, match="float32, float16 or bfloat16"):
        nb.roi_align_levels([lv[1].double()], torch.zeros(1, 5), 7, [0.25], 0)


def test_cpu_half_tensors_raise_nuhtc_error():
    import nuhtc_b200 as nb
    for dt in (torch.float16, torch.bfloat16):
        x = torch.zeros(1, 64, 8, 8, dtype=dt)
        with pytest.raises(nb.NuhtcError):
            nb.roi_align(x, torch.zeros(1, 5), 7)
        with pytest.raises(nb.NuhtcError):
            nb.to_cg32(x)
        with pytest.raises(nb.NuhtcError):
            nb.stage_levels([x])
