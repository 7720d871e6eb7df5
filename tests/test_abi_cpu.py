"""CPU: the C-ABI library builds/loads and exports every symbol include/tgan_b200.h declares (no compute calls)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "tgan_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tgan_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_the_expected_surface():
    names = _declared()
    for must in ("tgan_gemm", "tgan_relattn_fwd", "tgan_relattn_bwd", "tgan_ln_fwd", "tgan_ln_bwd", "tgan_ce_fwd",
                 "tgan_gumbel_st_fwd", "tgan_embed_fwd", "tgan_pack_params", "tgan_adam_step"):
        assert must in names


def test_library_loads_and_exports_every_declared_symbol():
    from tgan_b200 import lib
    cdll = ctypes.CDLL(lib.LIB_PATH)
    for name in _declared():
        assert hasattr(cdll, name), f"{name} declared in include/tgan_b200.h but not exported"
    assert lib.version() >= 100
    assert lib.has_tcgen05()
    # the Python binding table covers the same surface
    assert set(_declared()) == set(lib.EXPORTS)


def test_sass_contains_blackwell_tensor_core_and_tma_instructions():
    """The built .so must contain tcgen05 (UTCHMMA), TMEM loads (LDTM) and TMA (UTMALDG) SASS for sm_100a."""
    import shutil
    import subprocess
    from tgan_b200 import lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        import pytest
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnemonic in sass, mnemonic


def test_product_path_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "transformer-gan_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                txt = open(os.path.join(dirpath, f)).read()
                assert "txl_oracle" not in txt and "ref_harness" not in txt and "import oracle" not in txt, f


def test_library_has_no_environment_or_build_switches():
    """The kernels a call runs depend only on its arguments: no environment variable read by the library or its
    binding, and no project macro that compiles a second variant of a kernel."""
    pkg = os.path.join(ROOT, "transformer-gan_b200")
    csrc = os.path.join(pkg, "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh")):
            txt = open(os.path.join(csrc, f)).read()
            assert "getenv(" not in txt, f
            assert not re.search(r"#\s*if(n?def|\s+defined)\W*TGAN_", txt), f
    assert "os.environ" not in open(os.path.join(pkg, "tgan_b200", "lib.py")).read()
