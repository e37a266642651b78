"""Recipe for the Felzenszwalb-Huttenlocher checker of tests/test_felzenszwalb_ref.py -- TEST INFRASTRUCTURE ONLY.

The PC masker path of the reference is Python; the only C/C++ of the reference that touches a
stage next to the path is the vendored Felzenszwalb-Huttenlocher segmentation under
prim/src/FelzenSegment of a checkout of the reference (header-only, no build system needed).
When PCM_REFERENCE_ROOT points at that checkout, the headers are compiled FROM WHERE THEY LIE
(the sources are not copied) together with oracle/felzen_ref_shim.cpp:

    g++ -O2 -shared -fPIC -I$PCM_REFERENCE_ROOT/prim/src/FelzenSegment oracle/felzen_ref_shim.cpp \
        -o oracle/_ref/libfelzen_ref.so

oracle/_ref/ is git-ignored; a library built there earlier is used as it is.  Without either,
oracle/felzen_fh_restated.cpp -- the published algorithm restated with the same arithmetic and the
same C entry points -- is built into oracle/_build/ instead, so the comparison runs from the
repository alone.
"""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = os.environ.get("PCM_REFERENCE_ROOT", "")
FELZEN_INC = os.path.join(REF_SRC, "prim", "src", "FelzenSegment")
SHIM = os.path.join(HERE, "felzen_ref_shim.cpp")
LIB = os.path.join(HERE, "_ref", "libfelzen_ref.so")
RESTATED = os.path.join(HERE, "felzen_fh_restated.cpp")
RESTATED_LIB = os.path.join(HERE, "_build", "libfelzen_fh_restated.so")
FLAGS = ["g++", "-O2", "-std=c++14", "-w", "-ffp-contract=off", "-shared", "-fPIC"]


def _compile(src, lib, extra, force):
    if force or not os.path.isfile(lib) or os.path.getmtime(lib) < os.path.getmtime(src):
        os.makedirs(os.path.dirname(lib), exist_ok=True)
        subprocess.run(FLAGS + extra + [src, "-o", lib], check=True)
    return lib


def build(force=False):
    """Returns (path of the checker library, True when it is the reference's own code)."""
    if REF_SRC and os.path.isfile(os.path.join(FELZEN_INC, "segment-graph.h")):
        return _compile(SHIM, LIB, ["-I", FELZEN_INC], force), True
    if os.path.isfile(LIB):
        return LIB, True
    return _compile(RESTATED, RESTATED_LIB, [], force), False


if __name__ == "__main__":
    print(build(force=True))
