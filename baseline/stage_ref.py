#!/usr/bin/env python
"""Stages the UNMODIFIED Python reference into baseline/_ref/ (git-ignored) so that bench.py and the tests
can run the reference's own code.  The reference is a separate project: its checkout is given by --src or
HZ_REFERENCE_ROOT.  Nothing is edited: the *.py files and tests/ are copied as they are; run/logs/ is created
because loggers.py:22 opens log files under <root>/run/logs at import time (SURVEY.md §8c,
BASELINE.md §4 step 1).

    python baseline/stage_ref.py [--src <checkout of the reference>]
"""

import argparse
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")


def stage(src=None, dst=DST):
    src = src or os.environ.get("HZ_REFERENCE_ROOT")
    if not src or not os.path.isdir(src):
        return False
    os.makedirs(dst, exist_ok=True)
    for name in sorted(os.listdir(src)):
        p = os.path.join(src, name)
        if name.endswith(".py") and os.path.isfile(p):
            shutil.copy2(p, os.path.join(dst, name))
    tests = os.path.join(src, "tests")
    if os.path.isdir(tests):
        os.makedirs(os.path.join(dst, "tests"), exist_ok=True)
        for name in os.listdir(tests):
            if name.endswith(".py"):
                shutil.copy2(os.path.join(tests, name), os.path.join(dst, "tests", name))
    os.makedirs(os.path.join(dst, "run", "logs"), exist_ok=True)
    return True


def available(dst=DST):
    return os.path.exists(os.path.join(dst, "harmonies_engine.py")) and os.path.isdir(os.path.join(dst, "run", "logs"))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default=os.environ.get("HZ_REFERENCE_ROOT"), help="checkout of the reference (default: $HZ_REFERENCE_ROOT)")
    a = ap.parse_args()
    ok = stage(a.src)
    print("staged" if ok else f"reference checkout not found (--src {a.src})", DST)
    sys.exit(0 if ok else 1)
