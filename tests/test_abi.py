"""CPU test: liby5obb.so loads and exports exactly what include/y5obb.h declares (no compute calls)."""
import ctypes
import re
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]


def _declared():
    txt = (ROOT / "include" / "y5obb.h").read_text()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return set(re.findall(r"\b(y5obb_[a-z0-9_]+)\s*\(", txt))


def test_library_exports_every_declared_symbol():
    from yolov5_obb_b200.build import build_lib
    so = build_lib()
    L = ctypes.CDLL(str(so))
    decl = _declared()
    assert len(decl) >= 6
    for name in decl:
        assert hasattr(L, name), f"{name} declared in include/y5obb.h but not exported"
    out = subprocess.run(["nm", "-D", "--defined-only", str(so)], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (y5obb_[a-z0-9_]+)", out))
    assert exported == decl, f"header/library mismatch: {exported ^ decl}"


def test_python_prototypes_cover_the_abi():
    from yolov5_obb_b200 import _lib
    assert set(_lib.PROTOTYPES) == _declared()
    L = _lib.lib()
    assert L.y5obb_abi_version() >= 1
    assert b"sm_100a" in L.y5obb_build_info()
    assert L.y5obb_nms_workspace_bytes(1000, 1, 1000) > 1000 * 24


def test_no_product_import_of_oracle():
    """The product package must never import the oracle (parity would be void)."""
    for p in (ROOT / "yolov5_obb_b200").rglob("*.py"):
        src = p.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), p


def test_devkit_cpp_symbols_exported():
    """include/y5obb_devkit.hpp: the DOTA devkit's `_poly_nms` / `_overlaps` are exported under the reference's own C++ names
    (the mangled names the reference's poly_nms_kernel.cu / poly_overlaps_kernel.cu objects define), so the devkit's .pyx
    modules link against liby5obb.so unchanged."""
    from yolov5_obb_b200.build import build_lib
    so = build_lib()
    out = subprocess.run(["nm", "-D", "--defined-only", "-C", str(so)], capture_output=True, text=True).stdout
    assert "_poly_nms(int*, int*, float const*, int, int, float, int)" in out
    assert "_overlaps(float*, float const*, float const*, int, int, int)" in out
    # the same mangled symbols as the reference's own objects define (nm -D of poly_nms_kernel.cu / poly_overlaps_kernel.cu
    # compiled by oracle/build_ref.build_polygpu)
    mangled = set(re.findall(r" T (_Z9_\w+)", subprocess.run(["nm", "-D", "--defined-only", str(so)],
                                                            capture_output=True, text=True).stdout))
    assert {"_Z9_poly_nmsPiS_PKfiifi", "_Z9_overlapsPfPKfS1_iii"} <= mangled
