"""CPU: the C-ABI library builds/loads and exports exactly what include/pv_b200.h declares."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "pv_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(pv_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_functions():
    names = _header_functions()
    assert "pv_conv3d_fwd" in names and "pv_clip_transform_fwd" in names and len(names) >= 15


def test_library_loads_and_exports_every_declared_symbol():
    from pytorchvideo_b200 import _lib
    lib = _lib.load()
    for name in _header_functions():
        assert hasattr(lib, name), "libpvb200.so does not export %s" % name
    assert lib.pv_abi_version() == 1
    # the ctypes table binds exactly the declared functions
    assert sorted(_lib.SIGNATURES) == _header_functions()


def test_exports_are_c_linkage():
    from pytorchvideo_b200 import _lib
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.lib_path()], capture_output=True, text=True).stdout
    exported = set(l.split()[-1] for l in out.splitlines() if l.strip())
    for name in _header_functions():
        assert name in exported


def test_no_device_is_reported_not_faked():
    import torch
    from pytorchvideo_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        _lib.require_device()


def test_struct_sizes_match_header():
    """ctypes mirrors must have the C layout (compile a tiny probe with gcc)."""
    from pytorchvideo_b200 import _lib
    probe = r'''
    #include <stdio.h>
    #include "pv_b200.h"
    int main(){ printf("%zu %zu %zu %zu %zu\n", sizeof(pv_clip_transform_desc), sizeof(pv_conv3d_desc),
                       sizeof(pv_pool3d_desc), sizeof(pv_attention_desc), sizeof(pv_clip_batch_desc)); return 0; }'''
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "p.c")
        open(c, "w").write(probe)
        exe = os.path.join(td, "p")
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe], check=True)
        sizes = [int(v) for v in subprocess.run([exe], capture_output=True, text=True).stdout.split()]
    assert sizes == [ctypes.sizeof(_lib.ClipTransformDesc), ctypes.sizeof(_lib.Conv3dDesc),
                     ctypes.sizeof(_lib.Pool3dDesc), ctypes.sizeof(_lib.AttentionDesc), ctypes.sizeof(_lib.ClipBatchDesc)]


def test_product_has_no_cpu_path():
    import torch
    import pytorchvideo_b200.models.hub as H
    from pytorchvideo_b200.transforms import FusedClipTransform
    m = H.x3d_xs().eval()
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 4, 160, 160))
    with pytest.raises(RuntimeError):
        FusedClipTransform(4)(torch.zeros(3, 8, 16, 16, dtype=torch.uint8))


def test_product_never_imports_oracle():
    bad = []
    for dp, _, fs in os.walk(os.path.join(ROOT, "pytorchvideo_b200")):
        for f in fs:
            if f.endswith(".py") and re.search(r"^\s*(from|import)\s+oracle\b", open(os.path.join(dp, f)).read(), re.M):
                bad.append(f)
    assert not bad


# Entry points that need no direct parity test of their own, with the reason.
NO_DIRECT_GPU_TEST = {
    "pv_abi_version": "library metadata, checked on the CPU by test_library_loads_and_exports_every_declared_symbol",
    "pv_last_error": "error text only; every failing call in the suite reports it",
    "pv_device_info": "device query; every GPU test calls it through _lib.require_device",
    "pv_launch_count": "a counter; smoke() checks it grows",
    "pv_conv3d_tcgen05_supported": "host predicate, asserted by the conv cases that pick the tensor-core route",
    "pv_conv3d_stem_rows_supported": "host predicate, exercised by Plan.emit_conv in the stem route cases",
    "pv_bottleneck_fused_supported": "host predicate, exercised by the lowering of the fused bottleneck block",
    "pv_zero_f32": "a stream-ordered cudaMemsetAsync",
    "pv_clip_transform_fwd": "single-clip transform, compared with the numpy oracle by smoke()",
    "pv_bottleneck_fused_fwd": "covered through compile_model in test_gpu_ops.py::test_fused_bottleneck_block",
}


def test_every_compute_entry_point_has_a_direct_gpu_test():
    """Every pv_* function of include/pv_b200.h is named by at least one tests/test_gpu_*.py, unless it is listed in
    NO_DIRECT_GPU_TEST with a reason: a new entry point without a test, or a stale list entry, fails here."""
    names = _header_functions()
    stale = sorted(set(NO_DIRECT_GPU_TEST) - set(names))
    assert not stale, "NO_DIRECT_GPU_TEST names functions the header no longer declares: %s" % stale
    texts = []
    tests_dir = os.path.join(ROOT, "tests")
    for f in sorted(os.listdir(tests_dir)):
        if f.startswith("test_gpu_") and f.endswith(".py"):
            texts.append(open(os.path.join(tests_dir, f)).read())
    untested = [n for n in names if n not in NO_DIRECT_GPU_TEST
                and not any(re.search(r"\b%s\b" % n, t) for t in texts)]
    assert not untested, "entry points without a direct GPU test: %s" % untested
