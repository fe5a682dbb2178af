"""C-ABI surface checks that need no GPU: the library loads, exports every symbol include/ofb200.h
declares, the Python binding covers all of them, the C++ drop-in header compiles against it with the
reference's call sites, and compute entry points fail loudly (no CPU fallback) without a device."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ofb200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ofb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol_and_abi_version():
    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"libofb200.so does not export {n}"
    assert sorted(_lib.SIGNATURES) == names, "Python binding and header disagree"
    assert lib.ofb_version() == 101


@pytest.mark.parametrize("npix,threads", [(0, 1), (1, 1), (15, 2), (16, 1), (1000003, 3), (2 * 1920 * 1080, 4)])
def test_c3_extract_host(npix, threads):
    """Host-side extraction of channel 0 (what the batched host entry point does with ofb_ctx_set_host_threads): pure
    host code, no device involved."""
    import numpy as np
    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    rng = np.random.default_rng(npix + threads)
    src = rng.integers(0, 256, size=(npix, 3), dtype=np.uint8)
    dst = np.full(npix + 32, 0xAB, np.uint8)  # guard bytes behind the output
    rc = lib.ofb_c3_extract_host(src.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), npix, threads)
    assert rc == 0, lib.ofb_last_error()
    assert np.array_equal(dst[:npix], src[:, 0])
    assert (dst[npix:] == 0xAB).all()
    assert lib.ofb_c3_extract_host(None, dst.ctypes.data_as(C.c_void_p), npix, threads) != 0
    assert lib.ofb_c3_extract_host(src.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p), npix, 0) != 0


def test_header_compiles_as_c():
    """The boundary is plain C: no C++ or torch types in the signatures."""
    r = subprocess.run(["gcc", "-std=c99", "-fsyntax-only", "-x", "c", HEADER], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_dropin_header_compiles_with_reference_call_sites(tmp_path):
    """main.cu:209/250/260-style calls compile unchanged against include/OptFlowGpuB200.hpp."""
    src = tmp_path / "caller.cpp"
    src.write_text(
        '#include "OptFlowGpuB200.hpp"\n'
        "extern const float GAUS_KERNEL_3x3[];\n"
        "void frame(unsigned char** prev_pyramid, unsigned char** pyramid, float** flow_pyramid, int w, int h, int levels) {\n"
        "  gpu::gauss_pyramid(pyramid, w, h, levels, GAUS_KERNEL_3x3, 3, 3);\n"
        "  for (int k = levels - 1; k >= 0; k--)\n"
        "    gpu::calc_opt_flow(prev_pyramid[k], pyramid[k], w >> k, h >> k, flow_pyramid, k, levels);\n"
        "}\n"
        "void stages(const unsigned char* s, float* a, float* b, float** fp, const float* m, int w, int h) {\n"
        "  gpu::conv_3ch_1ch_tiled_uchar_float(s, w, h, a, m, 3, 3);\n"
        "  gpu::srm_1ch_float(a, a, w, h, 19, 19, b);\n"
        "  gpu::inverse_matrix_float(a, a, a, b, b, fp, 0, w, h);\n"
        "}\n")
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_no_cpu_fallback_without_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from cuda_optical_flow_2_b200 import Context, OfbError

    with pytest.raises(OfbError) as e:
        Context(0)
    assert e.value.code == 2 and "no CPU fallback" in str(e.value)


def test_null_context_is_rejected():
    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    assert lib.ofb_ctx_destroy(None) == _lib.OFB_ERR_INVALID
    assert b"NULL" in lib.ofb_last_error()
    p = _lib.OfbParams(64, 64, 1, 9, 2, 1.0, 1)
    assert lib.ofb_flow_pairs_device(None, C.byref(p), None, None, 64, 4096, None, None, None) == _lib.OFB_ERR_INVALID


def test_product_package_never_imports_the_oracle():
    """The product path must not route through oracle/ (it is test infrastructure)."""
    pkg = os.path.join(ROOT, "cuda_optical_flow_2_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "lk_oracle" not in text and "liblkoracle" not in text and "import oracle" not in text and \
                    "from oracle" not in text, f"{f} references the oracle"
    r = subprocess.run([sys.executable, "-c",
                        "import sys; sys.path.insert(0, %r); import cuda_optical_flow_2_b200; "
                        "print(any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules))" % ROOT],
                       capture_output=True, text=True)
    assert r.stdout.strip() == "False", r.stderr
