"""Stage the UNMODIFIED reference under oracle/_ref/ (TEST / BASELINE INFRASTRUCTURE ONLY).

The reference (hahnyuan/PTQ4ViT) is pure Python with no setup.py / pyproject, so "installing" it is a copy of its
importable packages from the tree named by $PTQ4VIT_REFERENCE.  oracle/_ref/ is git-ignored (never part of this
repository's history).  It is used by
  * tests/golden/make_*golden.py  -- the reference's outputs the parity tests compare against,
  * bench.py                      -- `--impl reference` (CPU arm) and the `reference_gpu` comparator (both fall back
                                     to the oracle's restatement where the reference is not staged).
Nothing under ptq4vit_b200/ and no test imports it.

    PTQ4VIT_REFERENCE=<reference tree> python oracle/stage_ref.py
"""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEST = os.path.join(ROOT, "oracle", "_ref")
PACKAGES = ("quant_layers", "utils", "configs")


def stage(src=None, quiet=False):
    """Copy the reference's importable packages; returns DEST, or None when no reference tree is available."""
    src = src or os.environ.get("PTQ4VIT_REFERENCE", "")
    if not src or not os.path.isdir(os.path.join(src, "quant_layers")):
        return DEST if os.path.isdir(os.path.join(DEST, "quant_layers")) else None
    os.makedirs(DEST, exist_ok=True)
    for pkg in PACKAGES:
        dst = os.path.join(DEST, pkg)
        if os.path.isdir(dst):
            shutil.rmtree(dst)
        shutil.copytree(os.path.join(src, pkg), dst, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
        for d, _, files in os.walk(dst):             # the source tree may be read-only: keep the copy removable
            os.chmod(d, 0o755)
            for f in files:
                os.chmod(os.path.join(d, f), 0o644)
    with open(os.path.join(DEST, "STAGED_FROM"), "w") as f:
        f.write(src + "\n")
    if not quiet:
        print(f"staged {', '.join(PACKAGES)} from {src} into {DEST}")
    return DEST


if __name__ == "__main__":
    sys.exit(0 if stage() else 1)
