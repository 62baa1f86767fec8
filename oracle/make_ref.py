"""Recipe for oracle/_ref: a runnable copy of the reference's environment path for the GPU box (TEST INFRASTRUCTURE ONLY).

    MARLSC_REFERENCE_ROOT=<marl-sc checkout> python oracle/make_ref.py      # also run by __graft_entry__.build()

The reference is pure Python, so "building" it means copying the modules its env step needs, unmodified, from the checkout
named by MARLSC_REFERENCE_ROOT into the git-ignored oracle/_ref/ (never committed; it can travel with the built .so files to
a machine without the checkout). bench.py --impl reference and the cpu_baseline leg then time the reference's own
InventoryEnvironment (src/environment/envs/multi_env.py) instead of the oracle port. Nothing in the product imports it.
"""
from __future__ import annotations

import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("MARLSC_REFERENCE_ROOT", "")
OUT = os.path.join(HERE, "_ref")

# what InventoryEnvironment imports, transitively, inside the reference's own tree
TREES = ["src/environment", "src/config"]
FILES = ["src/__init__.py", "src/utils/__init__.py", "src/utils/seed_manager.py", "src/data/__init__.py",
         "src/data/preprocessor.py", "src/data/data_generator.py"]


def main() -> int:
    if not REF:
        print("make_ref: MARLSC_REFERENCE_ROOT is not set; keeping whatever oracle/_ref holds")
        return 0
    if not os.path.isdir(os.path.join(REF, "src", "environment")):
        print(f"make_ref: MARLSC_REFERENCE_ROOT={REF!r} is not a marl-sc checkout (no src/environment)", file=sys.stderr)
        return 1
    if os.path.isdir(OUT):
        shutil.rmtree(OUT)
    for t in TREES:
        shutil.copytree(os.path.join(REF, t), os.path.join(OUT, t), ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    for f in FILES:
        src = os.path.join(REF, f)
        dst = os.path.join(OUT, f)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if os.path.exists(src):
            shutil.copy2(src, dst)
        else:
            open(dst, "w").close()                      # a package marker the reference does not have
    with open(os.path.join(OUT, "ORIGIN.txt"), "w") as fh:
        fh.write(f"Unmodified copies from {REF} (Jakoebly/marl-sc), made by oracle/make_ref.py. Not part of this repository.\n")
    n = sum(len(fs) for _, _, fs in os.walk(OUT))
    print(f"make_ref: {n} files -> {OUT}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
