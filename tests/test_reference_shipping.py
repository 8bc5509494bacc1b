"""oracle/_ref must be the reference byte for byte: every shipped source file against the SHA-256 digests of the
original's files (tests/golden/reference_sha256.json, taken from YannDubs/disentangling-vae @ f0452191), and the copy
must import as the reference's own `disvae` package.  CPU tests; they need the copy that build() ships when a checkout
of the reference is available (oracle/ship_reference.py)."""
import hashlib
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_sha256.json")


def _need_copy():
    if not os.path.isfile(os.path.join(DST, "main.py")):
        pytest.skip("oracle/_ref not shipped: build() found no checkout of the reference")


def test_shipped_reference_is_unmodified():
    _need_copy()
    want = json.load(open(DIGESTS))
    shipped = set()
    for base in ("disvae", "utils"):
        for d, _, files in os.walk(os.path.join(DST, base)):
            shipped.update(os.path.relpath(os.path.join(d, f), DST) for f in files if f.endswith(".py"))
    assert shipped == {k for k in want if k.startswith(("disvae/", "utils/"))}
    for rel, digest in want.items():
        with open(os.path.join(DST, rel), "rb") as fh:
            assert hashlib.sha256(fh.read()).hexdigest() == digest, rel
    assert len(want) > 15


def test_reference_imports_from_shipped_copy():
    _need_copy()
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); from oracle import reference_env as E; d = E.activate(%r); "
            "import disvae, os; assert os.path.realpath(disvae.__file__).startswith(os.path.realpath(d)); "
            "from disvae.training import Trainer; import main; print('ok')" % (ROOT, DST))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]
