import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# skani's own test_files/ directory: the full-size genomes a few oracle golden tests read (too large for tests/golden)
REF_TEST_FILES = os.environ.get("SKANI_TEST_FILES", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "slow: takes more than ~20 s on CPU")


def have_reference():
    return bool(REF_TEST_FILES) and os.path.isdir(REF_TEST_FILES)


needs_reference = pytest.mark.skipif(not have_reference(),
                                     reason="needs SKANI_TEST_FILES = skani's test_files directory (full-size genomes)")


def db_tool():
    """Path of the host-only database / FASTX helper (skani_b200/cli/skani_db_tool.cpp); built on demand (g++, no CUDA)."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "skani_b200", "skani-db-tool")
    src = [os.path.join(root, "skani_b200", "cli", f) for f in ("skani_db_tool.cpp", "sketch_db.hpp", "fastx.hpp")]
    if not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(f) for f in src):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-o", exe, src[0], "-lz"])
    return exe
