#!/usr/bin/env python
"""Records the reference's own outputs that tests/test_ref_pin.py compares the oracle against (tests/golden/ref_pin/*.npz, see tests/ref_golden.py).

Runs that test file with the reference build live (oracle/_ref/libvxref.so, made by `make -C oracle ref` where the original project's sources
are present): every value the reference side returns is written, and every comparison of the test is checked on the way.

    python tests/golden/make_ref_pin_golden.py
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, TESTS)
import ref_golden  # noqa: E402


def main():
    env = dict(os.environ, **{ref_golden.RECORD_ENV: "1"})
    rc = subprocess.run([sys.executable, "-m", "pytest", "-q", os.path.join(TESTS, "test_ref_pin.py")], env=env, cwd=os.path.dirname(TESTS)).returncode
    if rc != 0:
        sys.exit(f"test_ref_pin.py failed while recording (exit {rc}); the recordings under {ref_golden.GOLDEN_DIR} are not to be trusted")
    sizes = {f: os.path.getsize(os.path.join(ref_golden.GOLDEN_DIR, f)) for f in sorted(os.listdir(ref_golden.GOLDEN_DIR))}
    for f, n in sizes.items():
        print(f"{n:9d}  {f}")
    print(f"{sum(sizes.values()):9d}  total")


if __name__ == "__main__":
    main()
