"""CPU-side checks of the drop-in boundary: libfrr.so loads without a GPU and exports exactly the
entry points include/frr.h declares; the product refuses CPU tensors (no fallback)."""
import ctypes
import re
import subprocess

import numpy as np
import pytest
import torch

from faster_rcnn_pytorch_b200 import _lib, ops


def test_library_builds_loads_and_exports_every_declared_symbol_at_abi_version_3():
    from faster_rcnn_pytorch_b200 import build
    build.build()
    lib = _lib.load()
    names = _lib.declared_symbols()
    assert len(names) >= 8
    for n in names:
        assert hasattr(lib, n), n
        assert n in _lib.SIGNATURES, f"{n} declared in frr.h but not bound in _lib.SIGNATURES"
    assert set(_lib.SIGNATURES) == set(names)
    assert lib.frr_abi_version() == 3


_CTYPES = {"int": ctypes.c_int, "float": ctypes.c_float, "double": ctypes.c_double, "size_t": ctypes.c_size_t,
           "uint64_t": ctypes.c_uint64}


def _ctype(decl: str):
    """ctypes type of a C parameter or return type as frr.h spells it (a trailing parameter name is ignored)."""
    decl = decl.strip()
    if decl.startswith("const char*"):
        return ctypes.c_char_p
    if "*" in decl or decl.split()[0] == "frr_stream_t":
        return ctypes.c_void_p
    return _CTYPES[decl.split()[0]]


def test_signatures_match_the_header_prototypes():
    """Every prototype of include/frr.h against its _lib.SIGNATURES row: the restype and each argtype, in order."""
    with open(_lib.HEADER) as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)
    protos = re.findall(r"([A-Za-z_][\w ]*\**)\s*\b(frr_\w+)\s*\(([^)]*)\)\s*;", text)
    assert sorted(name for _, name, _ in protos) == _lib.declared_symbols()
    for ret, name, params in protos:
        params = params.strip()
        want = [] if params in ("", "void") else [_ctype(p) for p in params.split(",")]
        restype, argtypes = _lib.SIGNATURES[name]
        assert restype is _ctype(ret), f"{name}: restype {restype} vs {ret!r}"
        assert list(argtypes) == want, f"{name}: argtypes {argtypes} vs ({params})"


def test_library_reads_no_environment_variables():
    """Kernel and launch choices depend on the arguments and the device only, never on the process environment."""
    _lib.load()
    undefined = subprocess.run(["nm", "-D", "--undefined-only", _lib.LIB_PATH], check=True, capture_output=True,
                               text=True).stdout
    assert "getenv" not in undefined


@pytest.mark.parametrize("tune", [(128, 0, 0, 0), (0, 4096, 0, 0), (0, 0, 3, 0), (0, 0, 0, 64), (0, 0, -2, 0)])
def test_nms_sorted_settings_are_range_checked(tune):
    lib = _lib.load()
    rc = lib.frr_nms_sorted(None, None, 1, 0, 0.7, 0, None, None, None, 0, 0, *tune, 1, None)
    assert rc == -1 and b"frr_nms_sorted" in lib.frr_last_error()


def test_anchor_base_host_matches_oracle(oracle):
    assert np.array_equal(ops.anchor_base_table(), oracle.anchor_base_table())


def test_error_reporting_without_gpu():
    lib = _lib.load()
    rc = lib.frr_anchor_base_host(None, 16)
    assert rc == -1 and b"bad arguments" in lib.frr_last_error()
    with pytest.raises(ValueError):
        _lib.check(rc, "frr_anchor_base_host")


def test_ops_refuse_cpu_tensors():
    with pytest.raises(ValueError, match="no CPU path"):
        ops.nms_sorted(torch.zeros(1, 4, 4), 0.5)
    with pytest.raises(ValueError, match="no CPU path"):
        ops.topk_desc(torch.zeros(1, 4), 2)


def test_product_does_not_import_the_oracle():
    import os, re
    pkg = os.path.dirname(_lib.__file__)
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


def test_torch_library_ops_are_registered_with_fake_kernels():
    """torch.ops.frr.* exist with the torchvision schemas; the fake kernels give the output shapes on meta tensors
    (no GPU needed); no CPU kernel is registered (the region stage has no CPU path)."""
    import pytest
    import torch
    from faster_rcnn_pytorch_b200 import torch_ops  # noqa: F401  (registers the ops)
    feat = torch.empty((2, 8, 10, 12), device="meta")
    rois = torch.empty((5, 5), device="meta")
    out, arg = torch.ops.frr.roi_pool(feat, rois, 1.0, 7, 7)
    assert out.shape == (5, 8, 7, 7) and arg.shape == (5, 8, 7, 7) and arg.dtype == torch.int32
    assert torch.ops.frr.roi_align(feat, rois, 0.5, 7, 7, 2, False).shape == (5, 8, 7, 7)
    assert torch.ops.frr._roi_pool_backward(out, rois, arg, 1.0, 7, 7, 2, 8, 10, 12).shape == (2, 8, 10, 12)
    assert torch.ops.frr._roi_align_backward(out, rois, 1.0, 7, 7, 2, 8, 10, 12, 2, False).shape == (2, 8, 10, 12)
    r, c = torch.ops.frr.rpn_proposals(torch.empty((3, 90, 2), device="meta"), torch.empty((3, 90, 4), device="meta"),
                                       160, 256, 12000, 2000, 0.7, 0.001)
    assert r.shape == (3, 2000, 4) and c.shape == (3,) and c.dtype == torch.int32
    assert "Tensor dets, Tensor scores, float iou_threshold" in str(torch.ops.frr.nms.default._schema)
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.frr.roi_align(torch.zeros((1, 2, 4, 4)), torch.zeros((1, 5)), 1.0, 7, 7, 2, False)
