"""CPU tests of the drop-in boundary: libctcb200.so loads, exports every symbol include/ctcb200.h
declares, and its host-side (no-GPU) entry points behave.  No compute call is made here."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "ctcb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ctcb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    import _ctcb
    names = _declared()
    assert len(names) >= 18
    for n in names:
        assert hasattr(_ctcb.lib, n), "libctcb200.so does not export %s" % n
    assert set(names) == set(_ctcb.EXPORTS), "binding table and header disagree"
    assert _ctcb.lib.ctcb_version() >= 100


def test_header_cites_reference_interfaces():
    src = open(os.path.join(ROOT, "include", "ctcb200.h")).read()
    for cite in ("ctc_fast.pyx:13-152", "ctc_fast.pyx:154-187", "brnnet.py:10-277", "sgd.py:91-161",
                 "ctc_fast_blankforce.pyx:13-113", "rnnet.py:91-191", "nnet.py:57-113"):
        assert cite in src


def test_param_layout_matches_reference_stack():
    """Flat layout = the reference's stack order with its shapes (brnnet.py:38-41,66-72)."""
    import _ctcb
    cfg = _ctcb.BrnnConfig(41, 62, 512, 2, 1, 200, 32, 30, 0.0, 20.0)
    nt = _ctcb.lib.ctcb_brnn_num_tensors(ctypes.byref(cfg))
    assert nt == 2 * 3 + 4
    shapes, offs = [], []
    off, r, c = ctypes.c_int64(), ctypes.c_int32(), ctypes.c_int32()
    for i in range(nt):
        assert _ctcb.lib.ctcb_brnn_tensor_info(ctypes.byref(cfg), i, ctypes.byref(off), ctypes.byref(r), ctypes.byref(c)) == 0
        shapes.append((r.value, c.value)); offs.append(off.value)
    assert shapes == [(512, 41), (512, 1), (512, 512), (512, 1), (62, 512), (62, 1),
                      (512, 512), (1, 1), (512, 512), (1, 1)]
    assert all(o % 4 == 0 for o in offs) and offs == sorted(offs)
    n = _ctcb.lib.ctcb_brnn_param_count(ctypes.byref(cfg))
    assert n >= sum(a * b for a, b in shapes) and n % 4 == 0
    assert _ctcb.lib.ctcb_brnn_workspace_bytes(ctypes.byref(cfg)) > 0
    # temporalLayer >= numLayers+1 or <= 0 -> no temporal tensors
    cfg2 = _ctcb.BrnnConfig(41, 62, 512, 2, 0, 200, 32, 30, 0.0, 20.0)
    assert _ctcb.lib.ctcb_brnn_num_tensors(ctypes.byref(cfg2)) == 6
    # uni-directional: one recurrent matrix + its dummy bias (rnnet.py:57-65)
    cfg3 = _ctcb.BrnnConfig(41, 62, 512, 2, 1, 200, 32, 30, 0.0, 20.0, 1)
    assert _ctcb.lib.ctcb_brnn_num_tensors(ctypes.byref(cfg3)) == 8
    assert _ctcb.lib.ctcb_brnn_tensor_info(ctypes.byref(cfg3), 6, ctypes.byref(off), ctypes.byref(r), ctypes.byref(c)) == 0
    assert (r.value, c.value) == (512, 512)
    assert _ctcb.lib.ctcb_ctc_blankforce_workspace_bytes(4, 100, 61) == 4 * 100 * 61 * 8
    assert _ctcb.lib.ctcb_ctc_blankforce_workspace_bytes(4, 100, 1025) == 0


def test_error_reporting():
    import _ctcb
    cfg = _ctcb.BrnnConfig(41, 62, 512, 2, 1, 200, 32, 30, 0.0, 20.0)
    rc = _ctcb.lib.ctcb_brnn_tensor_info(ctypes.byref(cfg), 99, None, None, None)
    assert rc == -1 and b"out of range" in _ctcb.lib.ctcb_last_error()
    with pytest.raises(ValueError):
        _ctcb.check(rc)
    bad = _ctcb.BrnnConfig(0, 62, 512, 2, 1, 200, 32, 30, 0.0, 20.0)
    h = ctypes.c_void_p()
    assert _ctcb.lib.ctcb_brnn_create(ctypes.byref(bad), ctypes.byref(h)) == -1
    assert _ctcb.lib.ctcb_ctc_workspace_bytes(4, 100, 600) == 0          # > 511 labels: unsupported
    # the CTC kernel selector takes 0..4 (automatic, warp, pair, par, ckpt) and nothing else
    assert _ctcb.lib.ctcb_debug_set_ctc_kernel(7) == -1 and b"not in 0..4" in _ctcb.lib.ctcb_last_error()
    assert _ctcb.lib.ctcb_debug_set_ctc_kernel(0) == 0
    # fp64 trellis rows [T][64] + one (even-padded) word per 16-frame tile; two planes for small batches (alpha and beta)
    assert _ctcb.lib.ctcb_ctc_workspace_bytes(4, 100, 30) == 4 * (100 * 64 + 8) * 8 * 2
    assert _ctcb.lib.ctcb_ctc_workspace_bytes(1000, 100, 30) == 1000 * (100 * 64 + 8) * 8


def test_product_never_imports_the_oracle():
    """The product path must not route through oracle/ (or any CPU fallback)."""
    pkg = os.path.join(ROOT, "stanford-ctc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("# oracle", ""), "%s mentions the oracle" % f


_WITHOUT_CUDA = r'''
import os, sys
ROOT = %r
sys.path[:0] = [ROOT, os.path.join(ROOT, "stanford-ctc_b200")]
import numpy as np, pytest, torch
assert not torch.cuda.is_available()
import ctc_fast
p = np.asfortranarray(np.full((4, 5), 0.25))
with pytest.raises(RuntimeError):
    ctc_fast.ctc_loss(p, np.array([1, 2], dtype=np.int32))
with pytest.raises(ValueError):                       # reference contract checked before the device
    ctc_fast.ctc_loss(np.ascontiguousarray(p), np.array([1, 2], dtype=np.int32))
import nnets.brnnet as rnnet
with pytest.raises(RuntimeError):
    rnnet.NNet(5, 4, 8, 2, 10, temporalLayer=1)
'''


def test_product_fails_loudly_without_cuda():
    """In a process that sees no device (so that a machine with a GPU checks it too)."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, "-c", _WITHOUT_CUDA % ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
