"""Lays the drop-in over a copy of the reference tree, the way a maintainer of endiqq/Multi-Feature-ViT would deploy it:

    python multi-feature-vit_b200/tools/overlay.py /path/to/Multi-Feature-ViT /path/to/deploy

copies the reference checkout to /path/to/deploy and replaces, inside its moco_pretraining/moco/ directory, exactly the
modules INTEGRATION.md section 2 lists (vits.py, vits_returnftrs.py, model/module.py, model/crossvit_2vits_..._sum.py,
moco/builder_vit_mocov3structure_mocov2loss[_noprediction_q].py) by the ones of dropin/.  Everything else of the
reference - the main_*.py scripts, moco/loader.py, aihc_utils, training_tools, config - stays as it is, and the scripts
run unmodified (tests/test_reference_loop.py executes MAIN_CA's own train() that way).
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
DROPIN = os.path.join(PKG, "dropin")


def make_overlay(reference_root, dest):
    """dest = copy of reference_root with dropin/ laid over moco_pretraining/moco/.  Returns the directory that must be
    first on sys.path (the reference's own import root, SURVEY 3.0)."""
    if os.path.isdir(dest):
        shutil.rmtree(dest)
    shutil.copytree(reference_root, dest, ignore=shutil.ignore_patterns(".git", "__pycache__", "*.pyc"))
    target = os.path.join(dest, "moco_pretraining", "moco")
    for dirpath, _, files in os.walk(DROPIN):
        rel = os.path.relpath(dirpath, DROPIN)
        if "__pycache__" in rel:
            continue
        os.makedirs(os.path.join(target, rel), exist_ok=True)
        for f in files:
            if f.endswith(".py"):
                shutil.copy2(os.path.join(dirpath, f), os.path.join(target, rel, f))
    with open(os.path.join(target, "_mfvit_location.txt"), "w") as f:
        f.write(PKG + "\n")  # where libmfvit.so and the mfvit package live (read by _path.py)
    return target


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    print(make_overlay(sys.argv[1], sys.argv[2]))
