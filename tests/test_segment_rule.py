"""The angle rule of connected-component segmentation, on the host. cilantro_b200/csrc/segment_rule.hpp is its one
source: segment.cu compiles pair_passes for the device, cb_cloud_segment builds the interval ends with angle_bounds, and
tests/cpp/test_segment_rule.cpp compares the interval test with the evaluators' std::acos predicate for every float in
[-1, 1]. No GPU involved; the device side is tests/test_gpu_segment.py (exact parity with the oracle, dots at the
interval ends)."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "cilantro_b200", "csrc")


def test_angle_rule_against_acos_for_every_float(tmp_path):
    exe = str(tmp_path / "test_segment_rule")
    env = dict(os.environ)
    env.pop("CXX", None)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-pthread", "-Wall", "-I", CSRC,
                           os.path.join(ROOT, "tests", "cpp", "test_segment_rule.cpp"), "-o", exe], env=env)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=1800)
    print(out.stdout)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "all segment-rule checks passed" in out.stdout and "FAIL" not in out.stdout


def test_the_kernels_use_the_rule():
    """Every union / reachability kernel tests pairs through seg::pair_passes; segment.cu calls no acos of its own."""
    with open(os.path.join(CSRC, "segment.cu")) as f:
        src = re.sub(r"//[^\n]*", "", f.read())
    assert len(re.findall(r"seg::pair_passes\(", src)) == 3
    assert "acos" not in src and "seg::make_pair_rule(" in src
