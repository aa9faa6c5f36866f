"""Recipe: install the UNMODIFIED reference (lucidrains/x-clip, /root/reference) into oracle/_ref.

TEST / BENCH INFRASTRUCTURE ONLY.  The reference is a pure-Python package, so "building" it is a
`pip install --no-deps --target oracle/_ref` of a scratch copy of the read-only source tree
(setuptools writes build/ and *.egg-info next to setup.py, hence the copy under /tmp).  Nothing of
the reference is committed: oracle/_ref/ is git-ignored and travels to the GPU box with the tree,
like the built libxclip_b200.so.  Users of the result:

  * bench.py `cpu_baseline` / `--impl reference`  - the reference's own CLIP.forward + backward on
    the host cores (kind "reference"), and `gpu_eager_baseline` - the same unmodified module on
    the B200 in eager PyTorch (the only GPU path the reference has, SURVEY.md 8d);
  * tests/golden/make_golden.py imports the reference straight from /root/reference instead.

    python oracle/build_ref.py            # no-op when /root/reference is absent (GPU box)
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF_SRC = Path("/root/reference")
DEST = HERE / "_ref"


def available() -> bool:
    return (DEST / "x_clip" / "x_clip.py").exists()


def build(force: bool = False) -> bool:
    """Returns True when oracle/_ref holds the reference afterwards."""
    if available() and not force:
        return True
    if not os.path.isfile(REF_SRC / "setup.py"):    # absent or unreadable for this user
        return available()
    with tempfile.TemporaryDirectory(prefix="xclip_ref_src_") as tmp:
        src = Path(tmp) / "src"
        shutil.copytree(REF_SRC, src)
        for p in [src, *src.rglob("*")]:        # setup.py writes build/ into the copy's root
            p.chmod(p.stat().st_mode | 0o200)
        if DEST.exists():
            shutil.rmtree(DEST)
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
               "--target", str(DEST), str(src)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"pip install of the reference failed:\n{r.stdout}\n{r.stderr}")
    return available()


def import_reference():
    """-> the reference's `x_clip` module from oracle/_ref (raises if it was never built)."""
    if not available():
        raise RuntimeError("oracle/_ref is missing: run `python oracle/build_ref.py` in the build container")
    if str(DEST) not in sys.path:
        sys.path.insert(0, str(DEST))
    import x_clip  # noqa: F401  (the reference package, NOT x_clip_b200)
    return x_clip


if __name__ == "__main__":
    ok = build(force="-f" in sys.argv)
    print("oracle/_ref:", "ready" if ok else "unavailable (no /root/reference here)")
