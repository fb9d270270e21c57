#!/usr/bin/env python3
"""Records tests/golden/glsl_digests.json: the SHA-256 (tests/glsl_cases.py digest) of the compiled shaders' output on
every input that the comparisons of tests/test_oracle_vs_glsl.py and tests/test_oracle_vs_glsl_compute.py feed them, so
that those comparisons run on machines without the reference checkout too.  It runs those two test modules with
PT_RECORD_GLSL_DIGESTS=1.

With oracle/_ref/libglsl_ref.so and libglsl_comp_ref.so built, the digests are of the libraries' outputs.  Without them
they are of the oracle's outputs, which is right only for an oracle that passed every live comparison bit for bit.  The
committed file was recorded that way, from an oracle unchanged since the commit at which all of them passed with zero
differing records (DESIGN.md §4).
"""
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)


def main():
    os.environ["PT_RECORD_GLSL_DIGESTS"] = "1"
    path = os.path.join(HERE, "glsl_digests.json")
    if os.path.exists(path):
        os.remove(path)
    rc = pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(TESTS, "test_oracle_vs_glsl.py"),
                      os.path.join(TESTS, "test_oracle_vs_glsl_compute.py")])
    print(path, os.path.getsize(path), "bytes")
    sys.exit(rc)


if __name__ == "__main__":
    main()
