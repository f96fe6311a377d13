"""CPU suite: libssb.so loads and exports every symbol include/ssb.h declares
(no compute calls without a GPU), and the host-side logic around it."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from strongsort_yolo_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def lib_dbg(lib):
    from strongsort_yolo_b200 import _lib
    return _lib.load(debug=True)


def _declared(header="ssb.h"):
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ssb_[a-z0-9_]+)\s*\(", src)))


def _exported(path):
    import subprocess
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    return sorted({ln.split()[-1] for ln in out.splitlines() if ln.split()[-1].startswith("ssb_") and " T " in ln})


def test_exports_match_header(lib):
    """libssb.so exports exactly the extern "C" entry points include/ssb.h declares -- the baselines and
    diagnostics of include/ssb_debug.h are NOT in the product library."""
    from strongsort_yolo_b200 import _lib
    names = _declared()
    assert names, "no declarations parsed from include/ssb.h"
    assert sorted(_lib.SYMBOLS) == names
    for n in names:
        assert hasattr(lib, n), f"libssb.so does not export {n}"
    extern_c = [n for n in _exported(_lib.LIB_PATH) if not n.startswith("_Z")]
    assert sorted(set(extern_c) & set(_lib.DEBUG_SYMBOLS)) == []
    assert set(names) <= set(extern_c)


def test_debug_library_exports_the_debug_header(lib_dbg):
    from strongsort_yolo_b200 import _lib
    dbg = [n for n in _declared("ssb_debug.h") if n not in _declared()]
    assert sorted(_lib.DEBUG_SYMBOLS) == dbg
    for n in _lib.SYMBOLS + dbg:
        assert hasattr(lib_dbg, n), f"libssb_dbg.so does not export {n}"


def test_config_and_workspace_sizing(lib):
    from strongsort_yolo_b200 import _lib
    cfg = _lib.SsbConfig()
    lib.ssb_default_config(ctypes.byref(cfg))
    assert (cfg.max_dist, cfg.max_iou_distance, cfg.n_init, cfg.max_age, cfg.nn_budget) == \
        (0.2, 0.7, 3, 30, 100)
    assert abs(cfg.mc_lambda - 0.995) < 1e-15 and abs(cfg.ema_alpha - 0.9) < 1e-15
    n = lib.ssb_workspace_bytes(ctypes.byref(cfg))
    # gallery ring dominates: S * B * D * 4 bytes
    assert n > cfg.max_tracks * cfg.nn_budget * cfg.feat_dim * 4
    cfg.feat_dim = 7
    assert lib.ssb_workspace_bytes(ctypes.byref(cfg)) < 0
    assert b"feat_dim" in lib.ssb_last_error()


def test_weight_packing_matches_kernel_walk(lib_dbg, state_dict):
    from strongsort_yolo_b200 import weights
    lib = lib_dbg                                    # the fp32 blob belongs to the SIMT baseline
    tensors = weights.fold(state_dict)
    blob, sizes = weights.pack(tensors)
    n = lib.ssb_reid_num_tensors()
    assert n == len(tensors)
    want = (ctypes.c_int64 * n)()
    lib.ssb_reid_tensor_sizes(want)
    np.testing.assert_array_equal(np.asarray(list(want)), sizes)
    assert blob.size == int(((sizes + 3) & ~3).sum())


def test_bn_fold_matches_unfolded_oracle(state_dict):
    """Folding BN into conv (weights.fold) reproduces the oracle's conv->BN."""
    import torch
    import torch.nn.functional as F
    from strongsort_yolo_b200 import weights
    t = dict(weights.fold(state_dict))
    x = torch.randn(2, 3, 32, 16)
    w = torch.as_tensor(t["stem.w"]).permute(3, 2, 0, 1).contiguous()   # -> [co,ci,kh,kw]
    y = F.conv2d(x, w, torch.as_tensor(t["stem.b"]), stride=2, padding=3)
    sd = {k: torch.as_tensor(v) for k, v in state_dict.items()}
    r = F.conv2d(x, sd["conv1.conv.weight"], None, stride=2, padding=3)
    r = F.batch_norm(r, sd["conv1.bn.running_mean"], sd["conv1.bn.running_var"],
                     sd["conv1.bn.weight"], sd["conv1.bn.bias"], False, 0.0, 1e-5)
    np.testing.assert_allclose(y.numpy(), r.numpy(), rtol=1e-4, atol=1e-5)


def test_no_cpu_fallback():
    """Without a CUDA device the tracker refuses to construct.  The devices are hidden from a child process, so
    the check also runs on a machine that has a GPU."""
    code = (f"import sys\nsys.path.insert(0, {ROOT!r})\n"
            "from strongsort_yolo_b200 import _lib\n"
            "from strongsort_yolo_b200.strong_sort import StrongSORT\n"
            "try:\n"
            "    StrongSORT()\n"
            "except _lib.SsbError:\n"
            "    raise SystemExit(0)\n"
            "raise SystemExit('StrongSORT() constructed without a CUDA device')\n")
    p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
