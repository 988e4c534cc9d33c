"""CPU: the library build compiles every CUDA source and its rebuild digest covers every header a source includes, so
an edit to any of them rebuilds liboo_b200.so instead of leaving a stale library in place."""
import glob
import os
import re

from auto_oo_b200 import build


def test_every_source_is_compiled():
    found = sorted(os.path.basename(p) for p in glob.glob(os.path.join(build.CSRC, "*.cu")))
    assert sorted(build.SOURCES) == found


def test_every_included_header_is_in_the_digest():
    digested = {os.path.realpath(h) for h in build.HEADERS}
    for path in glob.glob(os.path.join(build.CSRC, "*.cu")) + glob.glob(os.path.join(build.CSRC, "*.cuh")):
        assert path.endswith(".cu") or os.path.realpath(path) in digested, path
        with open(path) as f:
            for inc in re.findall(r'^\s*#\s*include\s+"([^"]+)"', f.read(), re.M):
                header = os.path.realpath(os.path.join(os.path.dirname(path), inc))
                assert header in digested, (os.path.basename(path), inc)
