"""CPU: the C-ABI library loads and exports every symbol include/ugnet.h declares; the ctypes mirrors have the
sizes the header implies; the product path refuses to run without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import pytest
import torch

import ugnet_b200  # noqa: F401
from ugnet_b200 import engine as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "ugnet.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ug_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = E.load_library()
    declared = _header_functions()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in ugnet.h but not exported"
    assert sorted(E.EXPORTED_SYMBOLS) == declared
    assert lib.ug_version() == 100


def test_null_handle_is_rejected_not_crashing():
    lib = E.load_library()
    assert lib.ug_conv(None, None, None) != 0
    assert lib.ug_program_run(None, None, None) != 0
    assert lib.ug_last_error(None) == b"null handle"


def test_op_union_is_large_enough():
    assert ctypes.sizeof(E.Op) >= ctypes.sizeof(E.ConvDesc) + 8
    assert ctypes.sizeof(E.ConvDesc) % 8 == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    with pytest.raises(RuntimeError):
        E.Engine(0)
    from ugnet_b200.nets import UNetTaskAligWeight
    m = UNetTaskAligWeight(3, 1).eval()
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 224, 224))
    from ugnet_b200.googlenet import GoogLeNetClassifier
    with pytest.raises(RuntimeError):
        GoogLeNetClassifier(6).eval()(torch.zeros(1, 3, 224, 224))


def test_train_mode_is_rejected():
    from ugnet_b200.nets import UNetTaskAligWeight
    with pytest.raises(RuntimeError):
        UNetTaskAligWeight(3, 1).train()(torch.zeros(1, 3, 224, 224))


def test_product_package_never_touches_the_oracle_or_the_reference():
    """The oracle is test infrastructure: nothing under the shipped package may import it, read /root/reference, or
    fall back to a CPU / library implementation of the path (torch.nn.functional convolutions, cuDNN, Triton)."""
    pkg = os.path.join(ROOT, "unet-goolenet_b200")
    bad = []
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if not fn.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                continue
            src = open(os.path.join(dirpath, fn), encoding="utf-8").read()
            rel = os.path.relpath(os.path.join(dirpath, fn), ROOT)
            for pat in (r"^\s*(from|import)\s+oracle\b", r"/root/reference", r"\bimport\s+triton\b", r"torch\.compile\(",
                        r"F\.conv2d\(", r"\bcudnn[A-Z]\w*\(", r"\bcublas[A-Z]\w*\("):
                if re.search(pat, src, flags=re.M):
                    bad.append((rel, pat))
    assert not bad, bad


def _dev_header_functions():
    src = open(os.path.join(ROOT, "include", "ugnet_dev.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ug_[a-z0-9_]+)\s*\(", src)))


def test_dev_library_keeps_its_hooks_out_of_the_product_library():
    lib, dev = E.load_library(), ctypes.CDLL(E.DEV_LIB_PATH)
    assert sorted(E.DEV_SYMBOLS) == _dev_header_functions()
    for name in E.DEV_SYMBOLS:
        assert hasattr(dev, name), f"{name} declared in ugnet_dev.h but not exported by libugnet_dev.so"
        assert not hasattr(lib, name), f"{name} leaked into the product library"
    assert dev.ug_conv_launch_info(None, None, None) != 0


def test_conv_instance_tables():
    """ug_conv_instances (host only): 3 activations for each GEMM kernel, the multi kernel's table (both kinds, told
    apart by `pair`, no row listed twice), the pair kernel's 3 epilogues."""
    dev = ctypes.CDLL(E.DEV_LIB_PATH)
    row = ctypes.c_int * 6
    tables = []
    for k in range(5):
        n = dev.ug_conv_instances(k, None, 0)
        rows = (row * n)()
        assert dev.ug_conv_instances(k, rows, n) == n
        tables.append([tuple(r) for r in rows])
    assert dev.ug_conv_instances(5, None, 0) < 0
    assert tables[0] == tables[1] == [(a, -1, -1, -1, -1, -1) for a in (E.ACT_NONE, E.ACT_RELU, E.ACT_GELU)]
    assert tables[2] == tables[3] and len(set(tables[2])) == len(tables[2])
    assert any(t[5] for t in tables[2]) and not all(t[5] for t in tables[2])
    assert [t[2] for t in tables[4]] == [E.EPI_STORE, E.EPI_OUTC, E.EPI_GATE]
