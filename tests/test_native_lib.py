"""CPU: the C-ABI library builds in-tree, loads, exports every symbol include/ssdgeom.h declares,
and the host layer fails loudly (no CPU fallback) when there is no CUDA device."""
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ssdgeom.h")


@pytest.fixture(scope="module")
def native():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "ssd-object-detection_b200"))
    import build_native
    build_native.build()
    from ssdgeom import _native
    return _native


def declared_symbols():
    text = open(HEADER).read()
    return sorted(set(re.findall(r"SSDG_API\s+[\w\s\*]+?\b(ssdg_\w+)\s*\(", text)))


def test_header_declares_the_api():
    syms = declared_symbols()
    for must in ("ssdg_match_encode", "ssdg_multibox_loss", "ssdg_detect", "ssdg_nms", "ssdg_prior_boxes",
                 "ssdg_encode", "ssdg_decode", "ssdg_iou_pairs"):
        assert must in syms
    assert len(syms) >= 30


def test_library_exports_every_declared_symbol(native):
    out = subprocess.run(["nm", "-D", "--defined-only", native.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (ssdg_\w+)", out))
    declared = set(declared_symbols())
    assert declared <= exported, declared - exported
    assert exported <= declared, exported - declared          # nothing undocumented leaks out


def test_ctypes_table_covers_every_symbol(native):
    assert set(native.PROTOTYPES) == set(declared_symbols())
    lib = native.lib()
    assert lib.ssdg_version() == 100
    assert native.status_string(0) == "ok"
    assert "targets" in native.status_string(native.ERR_TOO_MANY_GT)    # utils/bbox.py:50 wording
    assert "thresh" in native.status_string(native.ERR_THRESH)          # utils/bbox.py:51 wording


def test_sass_has_bulk_tma_and_no_legacy_tensor_ops(native):
    """The streaming kernels use 1-D bulk TMA (UBLKCP) + mbarriers (SYNCS); nothing on this path is a
    dense contraction, so no tensor-core instruction may appear."""
    out = subprocess.run(["cuobjdump", "-sass", native.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    sass = out.stdout
    assert "sm_100a" in sass or "SM100" in sass.upper()
    assert "UBLKCP" in sass
    assert "SYNCS" in sass
    assert "REDUX" in sass
    assert "HMMA" not in sass and "UTCHMMA" not in sass


def test_argument_errors_need_no_gpu(native):
    lib = native.lib()
    # argument validation happens before any CUDA call
    assert lib.ssdg_match_encode(None, 0, None, None, None, 1, None, 1, 1, 1, 0.5, None, None, None, None, None, None, 0, None) == native.ERR_ARG
    assert lib.ssdg_multibox_loss(None, None, None, None, None, 1, 1, 2, 3, None, None, None, None, None, None, 0, None) == native.ERR_ARG
    assert lib.ssdg_match_workspace_bytes(256, 8732, 100) > 0
    assert lib.ssdg_loss_workspace_bytes(256, 8732, 81) >= 256 * 8732 * 4
    assert lib.ssdg_detect_workspace_bytes(2, 8732, 81, 200) >= 2 * 80 * 8732 * 8
    with pytest.raises(AssertionError):
        native.check(native.ERR_THRESH)
    with pytest.raises(AssertionError):
        native.check(native.ERR_TOO_MANY_GT)
    with pytest.raises(ValueError):
        native.check(native.ERR_ARG)
    from ssdgeom import device as D
    for priority in (0, 2, "medium"):          # "high", "low" or None only
        with pytest.raises(ValueError):
            D.Stream(priority)


def test_no_cpu_fallback(native):
    if native.device_count() > 0:
        pytest.skip("a CUDA device is present")
    from ssdgeom.utils import bbox
    with pytest.raises(native.SsdgeomError):
        bbox.iou([10, 10, 2, 2], [10, 10, 2, 2])
    with pytest.raises(native.SsdgeomError):
        bbox.match_bbox(np.zeros(1, np.float32), np.array([[.5, .5, .2, .2]], np.float32),
                        np.array([[.5, .5, .2, .2], [.1, .1, .1, .1]]))


def test_reference_asserts_are_raised_on_the_host(native):
    from ssdgeom.utils import bbox
    pri = np.array([[.5, .5, .2, .2]])
    g = np.tile(np.array([[.5, .5, .2, .2]], np.float32), (2, 1))
    with pytest.raises(AssertionError):
        bbox.match_bbox(np.zeros(2, np.float32), g, pri)              # T > A
    with pytest.raises(AssertionError):
        bbox.match_bbox(np.zeros(1, np.float32), g[:1], pri, 0.0)     # thresh
    with pytest.raises(AssertionError):
        bbox.apply_anchor_box(g, pri)                                  # shape, utils/bbox.py:95


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "ssd-object-detection_b200", "ssdgeom")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle|import_module\([\"']oracle", src, re.M), \
                    os.path.join(dirpath, f)
