"""The C-ABI shared library loads and exports every symbol include/*.h declares; without a GPU it refuses to
create a context (no CPU fallback). No compute calls here."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(poppy_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(native_lib):
    from poppy_b200 import _lib
    names = _declared("poppy_cuda.h") + _declared("poppy_host.h")
    assert len(names) >= 30
    for n in names:
        assert hasattr(native_lib, n), f"{n} declared in include/ but not exported by libpoppy_cuda.so"
    assert sorted(_lib.CUDA_ABI_SYMBOLS) == _declared("poppy_cuda.h")
    assert sorted(_lib.HOST_ABI_SYMBOLS) == [n for n in _declared("poppy_host.h")]


def test_version_string(native_lib):
    assert b"sm_100a" in native_lib.poppy_cuda_version()


def test_create_without_gpu_fails_loudly(native_lib):
    if native_lib.poppy_cuda_device_count() > 0:
        pytest.skip("a GPU is present")
    from poppy_b200.renderer import MorphRenderer
    from poppy_b200._lib import PoppyCudaError
    with pytest.raises(PoppyCudaError) as e:
        MorphRenderer(64, 64, 4, 16, 32, 1)
    assert e.value.code == -1 and "no CPU fallback" in str(e.value)


def test_product_does_not_reference_the_oracle():
    """Nothing under poppy_b200/ or include/ may import, link or load anything under oracle/."""
    bad = []
    for base, _, files in os.walk(os.path.join(ROOT, "poppy_b200")):
        if os.path.basename(base) in ("build", "__pycache__"):
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h")):
                text = open(os.path.join(base, f), errors="replace").read()
                if re.search(r"\boracle\b", text) and "oracle" in text.replace("# oracle", ""):
                    if re.search(r"(import|from|include|CDLL|dlopen).*oracle", text):
                        bad.append(os.path.join(base, f))
    assert not bad, bad


def test_library_reads_no_environment_variables():
    """The native library and its integration layer have no hidden run-time switches: nothing under
    poppy_b200/csrc/, include/ or integration/ calls getenv."""
    bad = []
    for top in ("poppy_b200/csrc", "include", "integration"):
        for base, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".cu", ".cuh", ".cpp", ".hpp", ".h", ".c")):
                    path = os.path.join(base, f)
                    if re.search(r"\b(secure_)?getenv\s*\(", open(path, errors="replace").read()):
                        bad.append(os.path.relpath(path, ROOT))
    assert not bad, bad


def test_kernels_are_compiled_for_sm_100a(native_lib):
    import shutil
    import subprocess
    from poppy_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_conditioning_entry_points_fail_loudly_without_a_gpu(native_lib):
    """poppy_cuda_blur_margin / poppy_cuda_gabor_filter have no CPU fallback either (only checked where no GPU is visible)."""
    import numpy as np
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is visible")
    except ImportError:
        pass
    from poppy_b200 import api
    with pytest.raises(RuntimeError, match="no such CUDA device|CUDA"):
        api.blur_margin(np.zeros((40, 50, 3), np.uint8), (60, 50))
    with pytest.raises(RuntimeError, match="no such CUDA device|CUDA"):
        api.gabor_filter(np.zeros((40, 50, 3), np.float32))
