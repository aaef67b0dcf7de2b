"""Host-only: the PLY passthrough of the PointCloud3f shim (tests/cpp/test_ply.cpp) — round trips in ascii and
binary, a hand-written file with another property layout and a face element, append / clear, a missing file."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ply_passthrough(tmp_path):
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    exe = str(tmp_path / "test_ply")
    lib = os.path.join(ROOT, "cilantro_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_ply.cpp"), "-o", exe, "-L", lib, "-lcilantro_b200",
                           f"-Wl,-rpath,{lib}"], env=env)
    out = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "PLY checks passed" in out.stdout


def test_reads_the_reference_scans(tmp_path):
    """The reference's bundled scans (binary little endian; colours between xyz and the normals, an extra 'radius'
    property) through the shim reader, compared with a direct numpy parse of the same bytes. The file is a crop of
    examples/test_clouds/test.ply in its own layout (tests/golden/scan_crop.ply)."""
    import numpy as np

    scan = os.path.join(ROOT, "tests", "golden", "scan_crop.ply")
    import sys

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from golden.make_config1_fixture import read_test_ply

    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    exe = str(tmp_path / "test_ply")
    lib = os.path.join(ROOT, "cilantro_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_ply.cpp"), "-o", exe, "-L", lib, "-lcilantro_b200",
                           f"-Wl,-rpath,{lib}"], env=env)
    out = subprocess.run([exe, str(tmp_path), scan], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    lines = out.stdout.strip().splitlines()
    p, n, c = read_test_ply(scan)
    assert lines[0].split() == ["scan", str(p.shape[0]), "1", "1"]
    for ln in lines[1:]:
        f = ln.split()
        i = int(f[1])
        got = np.array([float(x) for x in f[2:5] + f[6:9] + f[10:13]], np.float32)
        want = np.concatenate([p[i], n[i], c[i]]).astype(np.float32)
        assert np.array_equal(got, want), (i, got, want)
