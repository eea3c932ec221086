"""Stage the UNMODIFIED reference files of the hot path under baseline/_ref/ so that bench.py's CPU
arm (`--impl reference`, `cpu_baseline`, the `parity` block) runs the reference's own PyTorch code
(models/nerf.py, models/rendering.py, losses.py) on the GPU box's host cores.

    python tools/stage_reference.py            # copies from $NERF_PL_REFERENCE or /root/reference

baseline/_ref/ is git-ignored: the reference's sources never enter this repository.  Nothing stages
them implicitly (the build does not), so without this step bench.py's CPU arm times the numpy port
(oracle/) and a clean checkout behaves the same on every machine.  The reference's only native dependency
on this path, `torchsearchsorted`, does not build against torch 2.x (SURVEY.md section 8c); bench.py
registers the same 3-line shim tests/golden/make_golden.py uses (torch.searchsorted, verified
bit-identical on the reference's own test grid) before importing the staged modules.
"""
import hashlib
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILES = ["models/__init__.py", "models/nerf.py", "models/rendering.py", "losses.py", "LICENSE"]


def stage(ref=None, quiet=False) -> bool:
    ref = ref or os.environ.get("NERF_PL_REFERENCE", "/root/reference")
    if not os.path.isdir(ref):
        return False
    dst = os.path.join(ROOT, "baseline", "_ref")
    manifest = {}
    for rel in FILES:
        src = os.path.join(ref, rel)
        out = os.path.join(dst, rel)
        os.makedirs(os.path.dirname(out), exist_ok=True)
        shutil.copyfile(src, out)
        manifest[rel] = hashlib.sha256(open(src, "rb").read()).hexdigest()
    with open(os.path.join(dst, "MANIFEST.json"), "w") as f:
        json.dump({"source": ref, "sha256": manifest}, f, indent=1)
    if not quiet:
        print(f"staged {len(FILES)} reference files into {dst}")
    return True


if __name__ == "__main__":
    sys.exit(0 if stage(sys.argv[1] if len(sys.argv) > 1 else None) else 1)
