#!/usr/bin/env python
"""Recipe for the reference arm of bench.py: puts the UNMODIFIED reference under baseline/_ref/ (git-ignored, not
gpurun-ignored, so it travels to the GPU box; nothing from it is ever committed).

  1. `pip install --no-index --no-build-isolation --no-deps --target baseline/_ref <copy of /root/reference>`
     (from a /tmp copy: the build writes egg-info into the source tree and /root/reference is read-only).
     Outcome here: the install SUCCEEDS but ships metadata only — the reference's setup.py uses find_packages() and its
     model/ directory has no __init__.py, so the wheel contains no module (its own scripts do
     sys.path.insert(0, 'model') from a checkout instead).
  2. Therefore the modules the wheel leaves out are placed next to it byte for byte (model/*.py, main.py), which is
     what running the reference "from a checkout" means. bench.py --impl reference imports baseline/_ref/model/unet.py
     and drives FrameInterpolationUNet through its public API; no file is edited.

Run in the build container (where /root/reference exists): `python baseline/install_ref.py`. __graft_entry__.build()
calls it when /root/reference is present.
"""
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
REF = Path("/root/reference")
DST = ROOT / "baseline" / "_ref"


def reference_readable():
    """A reference this user may not read counts as absent: on a directory it cannot search, Path.exists() raises
    PermissionError rather than returning False."""
    try:
        return REF.exists() and os.access(REF, os.R_OK | os.X_OK)
    except PermissionError:
        return False


def main():
    if not reference_readable():
        print("baseline/install_ref.py: /root/reference is not present; keeping whatever baseline/_ref holds")
        return 0
    if DST.exists():
        shutil.rmtree(DST)
    with tempfile.TemporaryDirectory() as tmp:
        src = Path(tmp) / "reference"
        shutil.copytree(REF, src)
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps", "--quiet",
               "--find-links", "/opt/wheelhouse", "--target", str(DST), str(src)]
        rc = subprocess.run(cmd).returncode
        print(f"pip install --target baseline/_ref: exit code {rc}")
    (DST / "model").mkdir(parents=True, exist_ok=True)
    for rel in sorted(p.relative_to(REF) for p in list((REF / "model").glob("*.py")) + [REF / "main.py"]):
        shutil.copyfile(REF / rel, DST / rel)
        digest = hashlib.sha256((DST / rel).read_bytes()).hexdigest()[:16]
        print(f"  {rel}  sha256 {digest}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
