"""The C-ABI library loads without a GPU and exports exactly what include/xclip_b200.h declares."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def _declared():
    text = (ROOT / "include" / "xclip_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(xclip_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    from x_clip_b200 import _lib, build
    build.build()
    lib = _lib.load()
    names = _declared()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    for n in _lib.SIGNATURES:
        assert n in names, f"{n} bound in python but not declared in the header"


def test_abi_version_and_error_string_without_gpu():
    from x_clip_b200 import _lib
    lib = _lib.load()
    assert lib.xclip_abi_version() == 2
    assert isinstance(lib.xclip_last_error(), bytes)
    assert lib.xclip_nce_num_col_blocks(1024) == 4
    assert lib.xclip_nce_num_col_blocks(100) == 1


def test_no_cpu_fallback():
    """Without a CUDA device every compute entry fails loudly instead of falling back."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from x_clip_b200 import _lib, kernels
    rc = _lib.load().xclip_init()
    assert rc != 0 and _lib.load().xclip_last_error()
    with pytest.raises(_lib.XClipB200Error):
        kernels.gemm(torch.zeros(8, 8, dtype=torch.bfloat16), torch.zeros(8, 8, dtype=torch.bfloat16))


def test_product_never_imports_oracle():
    import re
    for f in (ROOT / "x_clip_b200").rglob("*.py"):
        assert not re.search(r"^\s*(from|import)\s+oracle|import_module\(.oracle", f.read_text(), re.M), f
        assert "oracle" not in f.read_text(), f   # not even mentioned: keeps the boundary obvious


def test_library_sass_is_tcgen05_tma_code():
    """The shipped kernels are sm_100a tcgen05 / TMEM / TMA code, not recompiled mma.sync / cp.async:
    the SASS of libxclip_b200.so must contain the Blackwell tensor-core, tensor-memory and bulk-tensor
    opcodes (UTCHMMA = tcgen05.mma, LDTM = tcgen05.ld, UTMALDG / UTMASTG = TMA tensor load / store,
    UTCBAR = tcgen05.commit) and the packed fp32x2 arithmetic of the GELU epilogues (FFMA2), and no
    legacy HMMA tensor instructions (profiles/r2_sass_histogram.md holds the full histogram)."""
    import shutil
    import subprocess
    from x_clip_b200 import _lib
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    try:
        sass = subprocess.run([exe, "-sass", str(_lib.LIB_PATH)], capture_output=True, text=True, timeout=300).stdout
    except (FileNotFoundError, subprocess.TimeoutExpired):
        import pytest
        pytest.skip("cuobjdump not available")
    assert "sm_100a" in sass
    for op, least in (("UTCHMMA", 100), ("LDTM", 50), ("UTMALDG", 50), ("UTMASTG", 10), ("UTCBAR", 20), ("FFMA2", 100)):
        assert sass.count(op) >= least, (op, sass.count(op))
    assert sass.count(" HMMA.") == 0
