"""The C-ABI boundary without a GPU: the library builds for sm_100a, loads, and exports exactly the symbols include/focoos_b200.h declares;
ops.load_library() gives every one of them the header's prototype and ops.py calls all of them; CudaBackend and its CPU mirror RefBackend
have the same interface; host-only entry points work; compute entry points refuse CPU tensors (no fallback)."""
import ctypes
import os
import re
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "focoos_b200.h")
LIB = os.path.join(ROOT, "focoos_b200", "lib", "libfocoos_b200.so")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g

    g.build()  # cached by a source hash; cross-compiles with nvcc when something changed
    return ctypes.CDLL(LIB)


def declared_symbols():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    return sorted(set(re.findall(r"\b(fb200_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported(lib):
    names = declared_symbols()
    assert len(names) >= 60
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/focoos_b200.h but not exported by {LIB}"
    nm = subprocess.run(["nm", "-D", "--defined-only", LIB], capture_output=True, text=True, check=True).stdout
    exported = sorted(set(re.findall(r" T (fb200_[a-z0-9_]+)", nm)))
    assert exported == names, (sorted(set(exported) - set(names)), sorted(set(names) - set(exported)))


def declared_param_counts():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    return {name: 0 if params.strip() in ("", "void") else params.count(",") + 1 for name, params in re.findall(r"\b(fb200_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text)}


def test_load_library_sets_header_prototypes(lib):
    from focoos_b200 import ops

    typed = ops.load_library()
    counts = declared_param_counts()
    assert sorted(counts) == declared_symbols() and list(ops.EXPORTED_SYMBOLS) == declared_symbols()
    for name, n in counts.items():
        assert len(getattr(typed, name).argtypes) == n, name
    assert typed.fb200_conv2d.argtypes[20] is ctypes.c_int64  # out_batch_stride
    assert typed.fb200_layernorm.argtypes[8] is ctypes.c_float  # eps
    assert typed.fb200_conv2d.argtypes[0] is ctypes.c_void_p and typed.fb200_conv2d.restype is ctypes.c_int
    for name in [n for n in counts if n.endswith("_workspace_bytes")]:
        assert getattr(typed, name).restype is ctypes.c_int64, name
    assert typed.fb200_last_error.restype is ctypes.c_char_p
    # nothing declared is left without a caller in the Python layer (fb200_version is the library's own version query, called below)
    src = open(os.path.join(ROOT, "focoos_b200", "ops.py")).read()
    assert [n for n in declared_symbols() if n not in src] == ["fb200_version"]


def test_backends_have_the_same_interface():
    import inspect

    from focoos_b200.ops import CudaBackend
    from oracle.ops_ref import RefBackend

    def public(cls):
        return {n: list(inspect.signature(f).parameters) for n, f in vars(cls).items() if callable(f) and not n.startswith("_")}

    assert public(CudaBackend) == public(RefBackend)


def test_host_only_entry_points(lib):
    from focoos_b200 import ops

    lib = ops.load_library()
    assert lib.fb200_version() >= 1
    assert lib.fb200_optim_workspace_bytes() > 0 and lib.fb200_detr_loss_workspace_bytes(7, 16, 300) > 0 and lib.fb200_col_workspace_bytes(256) > 0
    assert lib.fb200_conv_wgrad_tc_supported(16, 80, 80, 256, 80, 80, 256, 3, 3, 1, 1) == 1
    assert lib.fb200_conv_wgrad_tc_supported(16, 80, 80, 256, 40, 40, 256, 3, 3, 2, 1) == 1
    assert lib.fb200_conv_wgrad_tc_supported(16, 640, 640, 3, 320, 320, 32, 3, 3, 2, 1) == 0  # 3 channels: CUDA-core kernel
    # argument validation happens before any CUDA call: a null pointer is an error with a message, not a crash
    rc = lib.fb200_topk(None, 1, 10, 3, None, None, None)
    assert rc < 0 and b"topk" in lib.fb200_last_error()


def test_ops_refuse_cpu_tensors():
    from focoos_b200 import ops

    x = torch.zeros((1, 4, 4, 32))
    with pytest.raises(RuntimeError):
        ops.conv2d(x, torch.zeros((32, 1, 1, 32)))
    with pytest.raises(RuntimeError):
        ops.maxpool3x3s2(x)
