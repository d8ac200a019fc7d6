"""TEST / MEASUREMENT INFRASTRUCTURE ONLY.  Stage the unmodified reference for the CPU arm of bench.py.

    python oracle/stage_ref.py            # build container only (needs /root/reference)

`/root/reference` does not exist on the GPU box.  This recipe copies the reference's two Python packages
(`urban_planning/`, `khrylib/`: *.py files only, byte for byte) from where they lie into `oracle/_ref/`, which is
git-ignored (never part of the history: no reference source is committed) but NOT gpurun-ignored, so it travels with
the snapshot like the built `.so` files.  `bench.py --impl reference` then times the reference's OWN update step
(`tensorfy` + `AgentPG.value_loss` + `UrbanPlanningAgent.ppo_entropy_loss` + backward + `AgentPPO.clip_policy_grad` +
`torch.optim.Adam.step`, urban_planning_agent.py:322-337) on the box's host cores and reports
`cpu_baseline.kind = "reference"`; without `oracle/_ref` it falls back to the pinned oracle port (`kind = "port"`).
The geometry stack the reference imports transitively is stubbed by `oracle/ref_shim.py` exactly as for the golden
vectors.  `__graft_entry__.build()` runs this when `/root/reference` is present.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, "_ref")
PACKAGES = ("urban_planning", "khrylib")


def stage(src_root: str = "/root/reference", dest: str = DEST) -> dict:
    if not os.path.isdir(os.path.join(src_root, "urban_planning")):
        raise RuntimeError(f"reference tree not found at {src_root}")
    if os.path.isdir(dest):
        shutil.rmtree(dest)
    manifest = {}
    for pkg in PACKAGES:
        for dirpath, dirnames, filenames in os.walk(os.path.join(src_root, pkg)):
            dirnames[:] = [d for d in dirnames if d not in ("__pycache__",)]
            for fn in filenames:
                if not fn.endswith(".py"):
                    continue
                s = os.path.join(dirpath, fn)
                rel = os.path.relpath(s, src_root)
                d = os.path.join(dest, rel)
                os.makedirs(os.path.dirname(d), exist_ok=True)
                shutil.copyfile(s, d)
                with open(s, "rb") as f:
                    manifest[rel] = hashlib.sha256(f.read()).hexdigest()
    with open(os.path.join(dest, "MANIFEST.sha256"), "w") as f:
        for k in sorted(manifest):
            f.write(f"{manifest[k]}  {k}\n")
    return manifest


def staged_root() -> str | None:
    """Root to import the reference from: the copy staged under oracle/_ref, else None.  Run-time code reads only
    this copy, never the tree it was staged from."""
    if os.path.isdir(os.path.join(DEST, "urban_planning")):
        return DEST
    return None


if __name__ == "__main__":
    m = stage(sys.argv[1] if len(sys.argv) > 1 else "/root/reference")
    print(f"staged {len(m)} files -> {DEST}")
