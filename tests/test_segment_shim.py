"""ConnectedComponentExtraction3f<> through the C++ shims (include/cilantro/clustering/connected_component_extraction.hpp,
include/cilantro/core/common_pair_evaluators.hpp): the calls of the reference's examples/connected_component_extraction.cpp
(without the viewer and removeInvalidData) compile against the shims without a GPU, and on the GPU print the same labels
as cb_cloud_segment on the same downsampled cloud."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_segment_shim.cpp")
DEG2 = float(np.float32(2.0 * np.pi / 180.0))


def _build(tmp_path):
    exe = str(tmp_path / "test_segment_shim")
    env = dict(os.environ)
    env.pop("CXX", None)
    lib = os.path.join(ROOT, "cilantro_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"), SRC, "-o", exe,
                           "-L", lib, "-lcilantro_b200", f"-Wl,-rpath,{lib}"], env=env)
    return exe


def test_example_calls_compile_against_the_shims(cb, tmp_path):
    assert os.path.exists(_build(tmp_path))


def test_unsupported_evaluator_is_a_compile_error(tmp_path):
    src = tmp_path / "bad.cpp"
    src.write_text('#include <cilantro/clustering/connected_component_extraction.hpp>\n'
                   'struct Mine { bool operator()(size_t, size_t, float) const { return true; } };\n'
                   'int main() { cilantro::VectorSet3f p(3, 1); cilantro::ConnectedComponentExtraction3f<> c(p);\n'
                   '  c.segment(cilantro::RadiusNeighborhoodSpecification<float>(1.f), Mine()); }\n')
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode != 0 and "user-defined evaluators cannot cross the C ABI" in r.stderr


@pytest.mark.gpu
def test_example_through_the_shims_equals_the_c_abi(cb, ctx, tmp_path):
    from golden import make_ref_golden as ref_golden
    from golden.make_config1_fixture import read_test_ply

    out = subprocess.run([_build(tmp_path), ref_golden.CROP], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    labels = np.array([int(x) for x in out.stdout.split("labels")[1].split()], np.int64)
    p, nrm, col = read_test_ply(ref_golden.CROP)
    dp, dn, _ = cb.grid_downsample(ctx, p, 0.005, normals=nrm, colors=col)
    d = cb.Cloud(ctx, dp, dn)
    want = cb.segment(ctx, d, radius2=float(np.float32(0.02) * np.float32(0.02)), evaluator="normals", max_angle=DEG2,
                      min_size=100, max_size=dp.shape[0])
    d.close()
    assert np.array_equal(labels, want[0])
    assert f"{want[3]} components found" in out.stdout
