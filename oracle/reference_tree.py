"""Recipe for oracle/_ref/neddf: a writable copy of the parts of a ueda0319/neddf checkout that tests/test_harness.py
runs (the package, its Hydra configs, the bunny_smoke dataset and pretrained run).  build() stages it when the checkout
is present; the tests then read nothing outside this repository, and the reference's scripts write their logs into the
copy instead of the checkout.  oracle/_ref/ is a build product and stays out of git.

The checkout is NEDDF_REFERENCE_DIR, by default the one the oracle and the goldens under tests/golden were made from.
"""
import os
import shutil

SOURCE = os.environ.get("NEDDF_REFERENCE_DIR", "/root/reference")
DEST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "neddf")
PARTS = ("neddf", "config", os.path.join("pretrained", "bunny_smoke"), os.path.join("data", "bunny_smoke"))
_STAMP = ".staged_from"


def stage() -> bool:
    """Copy PARTS of SOURCE to DEST (again only when DEST came from elsewhere or is incomplete).  Without a readable
    checkout nothing changes, so a DEST staged earlier is kept.  Returns whether DEST is in place."""
    if not all(os.path.isdir(os.path.join(SOURCE, p)) for p in PARTS):
        return os.path.isfile(os.path.join(DEST, _STAMP))
    stamp = os.path.join(DEST, _STAMP)
    if os.path.isfile(stamp) and open(stamp).read() == os.path.abspath(SOURCE):
        return True
    if os.path.isdir(DEST):
        shutil.rmtree(DEST)
    for p in PARTS:
        shutil.copytree(os.path.join(SOURCE, p), os.path.join(DEST, p), copy_function=shutil.copyfile,
                        ignore=shutil.ignore_patterns("__pycache__"))
    for root, dirs, files in os.walk(DEST):  # the checkout may be read-only; copytree keeps directory modes
        for n in dirs + files:
            path = os.path.join(root, n)
            os.chmod(path, os.stat(path).st_mode | 0o200)
    os.chmod(DEST, os.stat(DEST).st_mode | 0o200)
    with open(stamp, "w") as f:
        f.write(os.path.abspath(SOURCE))
    return True
