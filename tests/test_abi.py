"""CPU-only checks of the drop-in boundary: the C-ABI library builds, loads, exports every symbol
that include/fbkst_b200.h declares, and the product path fails loudly without a GPU."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fbkst_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(fbkst_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib():
    from fbkst_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import importlib.util
        spec = importlib.util.spec_from_file_location(
            "fbkst_build", os.path.join(ROOT, "fbk-fairseq-st_b200", "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build()
    return _lib.load()


def test_header_declares_symbols():
    syms = declared_symbols()
    assert "fbkst_linear_bf16" in syms and "fbkst_ctc_compress" in syms and len(syms) >= 18


def test_library_exports_every_declared_symbol(lib):
    for name in declared_symbols():
        assert hasattr(lib, name), "libfbkst_b200.so does not export %s" % name


def test_binding_covers_every_declared_symbol():
    from fbkst_b200 import _lib
    bound = set(_lib.SIGNATURES) | set(_lib._RESTYPES) | {"fbkst_last_error"}
    assert set(declared_symbols()) == bound


def test_abi_version_and_error_string(lib):
    assert lib.fbkst_abi_version() == 1
    assert isinstance(lib.fbkst_last_error(), bytes)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback(lib):
    """Without a B200 the product path must raise, never fall back to CPU / PyTorch."""
    from fbkst_b200 import ops
    assert lib.fbkst_device_ok() == 0
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.layernorm(torch.zeros(4, 128), torch.ones(128), torch.zeros(128))


def test_argument_errors_do_not_need_a_gpu(lib):
    rc = lib.fbkst_linear_bf16(None, 8, None, 8, None, None, 0, None, 8, 4, 4, 8, 0, None, 0, None)
    assert rc == -1 and b"null operand" in lib.fbkst_last_error()
    rc = lib.fbkst_layernorm(1, 1, 1, 1, 0, 4, 100, ctypes.c_float(1e-5), None, 0, None)
    assert rc == -1 and b"unsupported D" in lib.fbkst_last_error()


def test_torch_custom_ops_are_registered_for_cuda_only():
    """torch.ops.fbkst.* exist (north_star: kernels exposed as PyTorch custom ops) and have no CPU
    kernel: the dispatcher refuses CPU tensors instead of falling back."""
    from fbkst_b200 import torch_ops
    for name in torch_ops.OPS:
        assert hasattr(torch.ops.fbkst, name), name
    with pytest.raises((NotImplementedError, RuntimeError), match="CPU"):
        torch.ops.fbkst.layernorm(torch.zeros(4, 128), torch.ones(128), torch.zeros(128), False, 1e-5)
