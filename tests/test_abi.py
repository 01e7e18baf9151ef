"""The C-ABI library loads on a CPU-only box and exports every symbol include/topoloss.h declares;
host-only entry points validate their arguments.  No compute call is made here."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "topoloss.h")


def _declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tl_[a-z_0-9]+)\s*\(", src)))


def test_header_declares_the_expected_entry_points():
    names = _declared()
    for must in ["tl_forward", "tl_backward", "tl_workspace_bytes", "tl_persistence_pairs", "tl_wasserstein",
                 "tl_last_error", "tl_version", "tl_status", "tl_set_option", "tl_pairs_workspace_bytes"]:
        assert must in names


def test_library_exports_every_declared_symbol():
    from dilabhelmholtzoct_b200 import _lib, build
    if not os.path.exists(build.LIB_PATH):
        build.build()
    L = ctypes.CDLL(build.LIB_PATH)
    for name in _declared():
        assert hasattr(L, name), f"{name} declared in topoloss.h but not exported"
    assert _lib.lib().tl_version() == _lib.ABI_VERSION
    assert set(_lib.SIGNATURES) <= set(_declared())


def test_distance_ops_have_one_entry_point_each():
    """ABI 5: each distance op takes its spacing as an argument (NULL: unit spacing); the _spaced twins are gone."""
    from dilabhelmholtzoct_b200 import _lib, build
    if not os.path.exists(build.LIB_PATH):
        build.build()
    L = ctypes.CDLL(build.LIB_PATH)
    assert _lib.ABI_VERSION == 5
    for op in ("tl_edt", "tl_hausdorff_dt_forward", "tl_surface_distances", "tl_signed_distance", "tl_boundary_forward"):
        assert op in _declared() and hasattr(L, op) and op in _lib.SIGNATURES, op
        gone = op + "_spaced"
        assert gone not in _declared() and not hasattr(L, gone) and gone not in _lib.SIGNATURES, gone


def _ws(L, B, C, H, W, d):
    ns, nc = ctypes.c_size_t(0), ctypes.c_size_t(0)
    rc = L.tl_workspace_bytes(B, C, H, W, d, ctypes.byref(ns), ctypes.byref(nc))
    return rc, ns.value, nc.value


def test_workspace_bytes_and_argument_errors():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    rc, ns, nc = _ws(L, 64, 14, 256, 256, 1)
    assert rc == 0 and ns > 0 and nc > 0
    rc, ns2, nc2 = _ws(L, 2, 14, 50, 50, 1)
    assert rc == 0 and ns2 < ns and nc2 < nc
    assert _ws(L, 2, 14, 50, 50, 2)[0] == -1      # feat_d = 2 is invalid on 2-D maps
    assert b"feat_d" in L.tl_last_error()
    assert _ws(L, 2, 14, 50, 60, 1)[0] == 0       # rectangular maps are fine (H rows of W pixels)
    assert _ws(L, 2, 14, 496, 512, 1)[0] == 0
    assert _ws(L, 0, 14, 50, 50, 1)[0] == -1
    assert L.tl_max_pairs(256, 256, 1) == 256 * 256 // 2 + 2
    with pytest.raises(ValueError):
        _lib.check(-1, "x")
    with pytest.raises(RuntimeError):
        _lib.check(-3, "x")


def test_workspace_is_small():
    """VERDICT r1 item 3: the headline shape needs <= 0.7 GB (was 3.41 GB), BASELINE configs[4]'s per-GPU shard
    (16 x 14 maps of 1024 x 1024) <= 6 GB (was 30.6 GB); the scratch part does not grow with the batch; the
    worst-case option restores the combinatorial maximum."""
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    assert L.tl_get_option(_lib.OPT_WORST_CASE_WORKSPACE) == 0
    rc, ns, nc = _ws(L, 64, 14, 256, 256, 1)
    assert rc == 0 and ns + nc <= 0.7e9, (ns, nc)
    assert ns >= 64 * 14 * 13000 * 24          # room for ~13 k pairs per map (iid noise: 12.9 k)
    rc, ns5, nc5 = _ws(L, 16, 14, 1024, 1024, 1)
    assert rc == 0 and ns5 + nc5 <= 6e9, (ns5, nc5)
    assert _ws(L, 8, 14, 256, 256, 1)[2] == nc  # scratch is per CTA, not per map
    try:
        assert L.tl_set_option(_lib.OPT_WORST_CASE_WORKSPACE, 1) == 0
        rc, nsw, ncw = _ws(L, 64, 14, 256, 256, 1)
        assert rc == 0 and nsw >= 64 * 14 * 2 * (256 * 256 // 2 + 2) * 24 and ncw >= nc
    finally:
        L.tl_set_option(_lib.OPT_WORST_CASE_WORKSPACE, 0)
    assert L.tl_set_option(99, 1) == -1


def test_product_has_no_cpu_path_and_never_imports_the_oracle():
    import torch
    import dilabhelmholtzoct_b200 as tlb
    x = torch.rand(2, 2, 8, 8)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.topo_loss(x, x, 0.1, feat_d=1)
    assert tlb.topo_loss(x, x, 0.0) == 0.0  # the reference's early-out returns a Python float
    pkg = os.path.join(ROOT, "dilabhelmholtzoct_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "topo_oracle" not in text, f


def test_fused_call_site_functions_have_no_cpu_path_either():
    """topo_loss_from_logits / resample / postprocess_masks (rows F1, F3): same rules as topo_loss --
    CUDA float32 only, the reference's early-out, argument errors raised on the host."""
    import torch
    import dilabhelmholtzoct_b200 as tlb
    x = torch.randn(2, 3, 8, 8)
    assert tlb.topo_loss_from_logits(x, x, 0.0, feat_d=1, interp=4) == 0.0
    with pytest.raises(ValueError, match="CUDA"):
        tlb.topo_loss_from_logits(x, x, 0.1, feat_d=1, interp=4)
    with pytest.raises(ValueError):
        tlb.topo_loss_from_logits(x, x[:, :2], 0.1, feat_d=1)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.resample(x, 4)
    with pytest.raises(ValueError, match="CUDA"):
        tlb.postprocess_masks(x, (6, 8), (5, 7), padded_size=8)


def test_resample_and_postprocess_argument_errors_from_the_library():
    from dilabhelmholtzoct_b200 import _lib
    L = _lib.lib()
    assert L.tl_resample_forward(None, 1, 8, 8, 4, 1, None, None) == -1 and b"null" in L.tl_last_error()
    assert L.tl_resample_forward(1, 0, 8, 8, 4, 1, 1, None) == -1
    assert L.tl_postprocess_forward(1, 1, 8, 8, 32, 40, 32, 16, 16, 1, None) == -1   # crop larger than the intermediate
    assert b"crop" in L.tl_last_error()
    assert L.tl_postprocess_backward(None, 1, 8, 8, 32, 32, 32, 16, 16, None, None) == -1
