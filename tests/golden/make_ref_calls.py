"""Generates tests/golden/ref_calls_*.npz: the answers of the reference's own code (oracle/_ref/) to every call the tests
below make into it (see tests/ref_replay.py).  Needs oracle/_ref/ built, i.e. `make -C oracle ref` with the reference
tree present; run from anywhere:  python tests/golden/make_ref_calls.py"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
MODULES = ["tests/test_reference_functors.py", "tests/test_lduops.py", "tests/test_limiters_cpu.py", "tests/test_mules_cpu.py",
           "tests/test_ref_golden.py"]

if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    from oracle import ref_ldu
    assert ref_ldu.available(), "oracle/_ref is not built: this script needs the reference tree"
    env = dict(os.environ, B200LDU_RECORD_REF="1")
    sys.exit(subprocess.call([sys.executable, "-m", "pytest", "-q", "-m", "not gpu", "-p", "no:cacheprovider", *MODULES],
                             cwd=ROOT, env=env))
