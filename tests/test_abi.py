"""CPU-side checks of the C-ABI boundary: the library builds for sm_100a, loads, and exports every
symbol that include/nxfx_b200.h declares (no compute calls without a GPU)."""

import ctypes
import pathlib
import re

ROOT = pathlib.Path(__file__).resolve().parent.parent


def declared_symbols():
    text = (ROOT / "include" / "nxfx_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(nxfx_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported(built_library):
    lib = ctypes.CDLL(str(built_library))
    names = declared_symbols()
    assert len(names) >= 25
    for name in names:
        assert hasattr(lib, name), f"{name} declared in nxfx_b200.h but not exported"


def test_binding_covers_header(built_library):
    from networks_fenicsx_b200 import _lib

    assert sorted(_lib.SIGNATURES) == declared_symbols()
    lib = _lib.load()
    assert lib.nxfx_abi_version() == 2


def test_create_fails_loudly_without_gpu(built_library):
    """No CPU fallback: without a CUDA device the product raises."""
    import pytest
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from networks_fenicsx_b200.device import Device

    with pytest.raises(RuntimeError, match="no usable CUDA device"):
        Device(0)
    import networks_fenicsx_b200 as nxfx

    G = nxfx.network_generation.make_tree(2, 1, 3)
    nm = nxfx.NetworkMesh(G, N=4)  # host analysis works without a GPU ...
    with pytest.raises(RuntimeError):
        nm.mesh.geometry.x  # ... anything numeric does not


def test_product_does_not_import_oracle():
    for path in (ROOT / "networks_fenicsx_b200").rglob("*.py"):
        text = path.read_text()
        assert "import oracle" not in text and "from oracle" not in text, path


def test_sass_is_sm100(built_library):
    import shutil
    import subprocess

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([cuobjdump, "-lelf", str(built_library)], capture_output=True, text=True).stdout
    assert "sm_100a" in out
