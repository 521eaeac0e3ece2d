"""CPU-only checks of the build entry points (include/gbwt_b200_build.h): the library exports what the header declares,
refuses an empty path set, and without a GPU refuses to build instead of falling back to the CPU."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_the_build_header():
    import gbwt_rs_b200 as gb
    text = open(os.path.join(ROOT, "include", "gbwt_b200_build.h")).read()
    names = sorted(set(re.findall(r"GBWT_B200_API\s+[^;(]*?\b(gbwt_b200_\w+)\s*\(", text)))
    assert names == ["gbwt_b200_build_image", "gbwt_b200_build_image_device"]
    lib = ctypes.CDLL(gb.LIBRARY)
    for name in names:
        assert hasattr(lib, name)


def test_no_paths_is_an_argument_error():
    import gbwt_rs_b200 as gb
    with pytest.raises(gb.GBWTError) as info:
        gb.build_image([])
    assert info.value.code == gb.E_ARGUMENT


def test_no_cpu_fallback_without_a_device():
    import gbwt_rs_b200 as gb
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("a GPU is present")
    with pytest.raises(gb.GBWTError) as info:
        gb.build_image([[2, 4, 6]])
    assert info.value.code == gb.E_NO_DEVICE
