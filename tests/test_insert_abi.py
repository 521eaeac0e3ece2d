"""CPU-only checks of the insertion entry points (include/gbwt_b200_insert.h): the library exports what the header declares,
with the documented argument order, the build header includes it, and a null index is refused without a GPU."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declarations():
    text = open(os.path.join(ROOT, "include", "gbwt_b200_insert.h")).read()
    out = {}
    for name, args in re.findall(r"GBWT_B200_API\s+int\s+(gbwt_b200_\w+)\s*\(([^;]*)\)\s*;", text):
        out[name] = [a.strip().split()[-1].lstrip("*").split("[")[0] for a in " ".join(args.split()).split(",")]
    return out


def test_library_exports_the_insert_header():
    import gbwt_rs_b200 as gb
    decl = declarations()
    assert sorted(decl) == ["gbwt_b200_insert_image", "gbwt_b200_insert_image_device"]
    lib = ctypes.CDLL(gb.LIBRARY)
    for name in decl:
        assert hasattr(lib, name)


def test_argument_order():
    decl = declarations()
    assert decl["gbwt_b200_insert_image"] == ["index", "nodes", "offsets", "n", "image", "len", "info"]
    assert decl["gbwt_b200_insert_image_device"] == ["index", "d_nodes", "d_offsets", "n", "stream", "image", "len", "info"]
    text = open(os.path.join(ROOT, "include", "gbwt_b200_insert.h")).read()
    assert "uint64_t info[6]" in text


def test_build_header_includes_it():
    text = open(os.path.join(ROOT, "include", "gbwt_b200_build.h")).read()
    assert '#include "gbwt_b200_insert.h"' in text


def test_null_index_is_an_argument_error():
    import gbwt_rs_b200 as gb
    lib = gb.library()
    image, ln = ctypes.c_void_p(), ctypes.c_size_t(0)
    assert lib.gbwt_b200_insert_image(None, None, None, 1, ctypes.byref(image), ctypes.byref(ln), None) == gb.E_ARGUMENT
    assert lib.gbwt_b200_insert_image_device(None, None, None, 1, None, ctypes.byref(image), ctypes.byref(ln), None) == gb.E_ARGUMENT
