"""CPU: the C-ABI library loads without a GPU and exports every symbol include/nuhtc_b200.h declares; the product
package never touches the oracle; ops refuse CPU tensors (no silent fallback)."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    hdr = open(os.path.join(ROOT, "include", "nuhtc_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(nuhtc_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    import nuhtc_b200
    from nuhtc_b200 import _lib
    names = _declared()
    assert len(names) >= 12
    assert set(names) == set(_lib.SIGNATURES), "header and ctypes table disagree"
    L = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(L, n), n
    assert _lib.lib().nuhtc_abi_version() == 1


def test_library_is_sm100a_native():
    from nuhtc_b200 import _lib
    nvcc = shutil.which("nvcc")         # the toolkit that built the library
    tool = shutil.which("cuobjdump") or (nvcc and shutil.which("cuobjdump", path=os.path.dirname(nvcc)))
    if not tool:
        pytest.skip("cuobjdump unavailable")
    out = subprocess.run([tool, "--list-elf", _lib.LIB_PATH], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "sm_100a" in out.stdout


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "nuhtc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "libnuhtc_oracle" not in src and "nuhtc_oracle.c" not in src, f


def test_ops_refuse_cpu_tensors():
    import nuhtc_b200 as nb
    with pytest.raises(nb.NuhtcError):
        nb.roi_align(torch.zeros(1, 64, 8, 8), torch.zeros(1, 5), 7)
    with pytest.raises(nb.NuhtcError):
        nb.nms(torch.zeros(2, 4), torch.zeros(2), 0.5)
    with pytest.raises(nb.NuhtcError):
        nb.paste_masks(torch.zeros(1, 1, 28, 28), torch.zeros(1, 4), 8, 8)
    with pytest.raises(nb.NuhtcError):
        nb.pack_masks(torch.zeros(1, 8, 8, dtype=torch.uint8))
    with pytest.raises(nb.NuhtcError):
        nb.merge_arrays(torch.zeros(3, 2, dtype=torch.float64), torch.tensor([0, 3]), torch.zeros(1, dtype=torch.float64))


def test_argument_validation_without_gpu():
    """bad arguments are rejected by the library before any CUDA call"""
    from nuhtc_b200 import _lib
    L = _lib.lib()
    assert L.nuhtc_roi_align_fwd(None, None, None, None, 0, 1, 64, 1, None, 1, 7, 7, 0, 1, 0, 56.0, 0, None, None, None) == -1
    assert b"L=0" in L.nuhtc_last_error()
    assert L.nuhtc_paste_masks(None, None, 1, 100, 100, 8, 8, 0.5, 1, None, None, None, None) == -1
    assert L.nuhtc_nms_workspace_bytes(5000, 16, 5000, 0) > 5000 * 79 * 8
    assert L.nuhtc_nms_workspace_bytes(0, 1, 0, 0) == 256


def test_argument_validation_of_the_later_entry_points():
    """contours / glue / dual paste: sizes and null pointers are rejected before any CUDA call; empty inputs are accepted"""
    import ctypes
    from nuhtc_b200 import _lib
    L = _lib.lib()
    F4 = ctypes.c_float * 4
    one, zero = F4(1, 1, 1, 1), F4(0, 0, 0, 0)
    assert L.nuhtc_mask_contours(None, None, None, -1, 64, 64, 8, None, None, None, None) == -1
    assert L.nuhtc_mask_contours(None, None, None, 4, 64, 64, 0, None, None, None, None) == -1        # max_pts < 1
    assert L.nuhtc_contour_rings(None, None, None, None, 3, 16, None, None) == -1                     # null pointers, n > 0
    assert L.nuhtc_contour_rings(None, None, None, None, 0, 16, None, None) == 0                      # nothing to do
    assert L.nuhtc_delta2bbox(None, 1, None, 5, zero, one, 64, 64, 16 / 1000, 1.0, None, None) == -1  # null pointers, K > 0
    assert L.nuhtc_delta2bbox(None, 1, None, 0, zero, one, 64, 64, 16 / 1000, 1.0, None, None) == 0
    assert L.nuhtc_delta2bbox(None, 1, None, 0, zero, one, 64, 64, 0.0, 1.0, None, None) == -1        # wh_ratio_clip must be > 0
    assert L.nuhtc_multiclass_candidates(None, 3, None, 6, None, 5, 4, 5, 0.05, None, None, None, None, None, None) == -1  # stride < 4
    assert L.nuhtc_detection_slots(None, None, None, 0, 10, None, None, None, None, 1.0, None, None, None, None, None, None, None, None) == -1
    assert L.nuhtc_tile_filter(None, None, None, 0, 0, 256, 256, 10, None, None) == 0
    assert L.nuhtc_keep_flags(None, None, None, 0, 10, 5, None, None) == -1                           # num_tiles < 1
    assert L.nuhtc_paste_masks_dense_bits(None, None, 2, 28, 28, 64, 60, 0.5, None, None, None, None, None) == -1   # width % 16
    assert b"multiple of 16" in L.nuhtc_last_error()
    assert L.nuhtc_paste_masks_dense_bits(None, None, 0, 28, 28, 64, 64, 0.5, None, None, None, None, None) == 0
