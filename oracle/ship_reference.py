#!/usr/bin/env python
"""Place the UNMODIFIED reference (YannDubs/disentangling-vae) inside the tree where the tests and the benchmark find it:
a checkout of it -> git-ignored oracle/_ref/.

The reference's sources never enter this repository's history; oracle/_ref/ is a build product that travels with the
working tree like the built .so.  The reference has no setup.py / pyproject.toml, so there is nothing to install; this
recipe copies the Python sources, `hyperparam.ini` and the licence verbatim instead (no edits --
`tests/test_reference_shipping.py` checks the copy against SHA-256 digests of the original files).

Where the reference checkout is, first match: $DISVAE_REFERENCE; `reference_path` in BASELINE.json (where the
reference this project was measured against is kept); a directory named `reference` next to this repository.

Used by: `bench.py --impl reference` / `--impl reference-cuda` (the reference's own Trainer on the host cores / on
the GPU through stock PyTorch eager) and `tests/test_main_gpu.py` (the reference's `main.py` driving this
repository's `disvae` package).  Run by `__graft_entry__.build()`, or:  python oracle/ship_reference.py
"""
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
ITEMS = ["disvae", "utils", "main.py", "main_viz.py", "hyperparam.ini", "LICENSE"]


def candidates():
    out = []
    if os.environ.get("DISVAE_REFERENCE"):
        out.append(os.environ["DISVAE_REFERENCE"])
    with open(os.path.join(ROOT, "BASELINE.json")) as fh:
        recorded = json.load(fh).get("reference_path")
    if recorded:
        out.append(recorded)
    out.append(os.path.join(os.path.dirname(ROOT), "reference"))
    return out


def find_checkout():
    for d in candidates():
        if os.path.isfile(os.path.join(d, "main.py")) and os.path.isfile(os.path.join(d, "disvae", "training.py")):
            return d
    return None


def _copy_tree(src, dst):
    """File contents only: the reference's checkout may be read-only, and copied modes would leave directories the
    next build() could not replace."""
    for d, dirs, files in os.walk(src):
        dirs[:] = [x for x in dirs if x != "__pycache__"]
        out = os.path.join(dst, os.path.relpath(d, src))
        os.makedirs(out, exist_ok=True)
        for f in files:
            if not f.endswith(".pyc"):
                shutil.copyfile(os.path.join(d, f), os.path.join(out, f))


def ship(verbose=True):
    ref = find_checkout()
    if ref is None:
        if verbose:
            print("no reference checkout in %s: keeping whatever oracle/_ref holds" % candidates())
        return os.path.isdir(os.path.join(DST, "disvae"))
    os.makedirs(DST, exist_ok=True)
    for it in ITEMS:
        src, dst = os.path.join(ref, it), os.path.join(DST, it)
        if os.path.isdir(src):
            if os.path.isdir(dst):
                shutil.rmtree(dst)
            _copy_tree(src, dst)
        else:
            shutil.copyfile(src, dst)
    if verbose:
        print("reference shipped from %s to %s" % (ref, DST))
    return True


if __name__ == "__main__":
    sys.exit(0 if ship() else 1)
