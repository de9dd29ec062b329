"""Runs one test in a child pytest whose CUDA runtime sees no device, so the checks of the no-GPU failure paths also run
on machines that have a GPU."""
import os
import subprocess
import sys


def rerun_without_gpu(test_file, name):
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "%s::%s" % (test_file, name)],
                       cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "1 passed" in r.stdout, (r.stdout[-3000:], r.stderr[-2000:])
