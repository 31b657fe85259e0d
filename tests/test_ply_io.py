"""include/pcpx/ply.hpp (host-only PLY reader / writer, SURVEY.md §8f rank 4) against the
reference's on-disk format: byte streams written by the UNMODIFIED reference writer
(tests/golden/ref_ply.npz, made by make_ply_fixtures.py) must be read back exactly, and the
writer must produce those same bytes.  Also the reference's real scans when PCP_REFERENCE
names a checkout of the reference."""
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(os.path.dirname(__file__), "golden", "ref_ply.npz")
FORMATS = {"ascii": "0", "binary_little_endian": "1", "binary_big_endian": "2"}


@pytest.fixture(scope="module")
def tool(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("ply") / "ply_tool")
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "ply_tool.cpp"), "-o", exe], check=True)
    return exe


@pytest.fixture(scope="module")
def fix():
    return np.load(FIX)


def read_flat(tool, ply_path, tmp_path):
    out = str(tmp_path / "flat.bin")
    rc = subprocess.run([tool, "read", ply_path, out]).returncode
    raw = open(out, "rb").read()
    n, m = struct.unpack("<QQ", raw[:16])
    xyz = np.frombuffer(raw, np.float32, 3 * n, 16).reshape(-1, 3)
    nrm = np.frombuffer(raw, np.float32, 3 * m, 16 + 12 * n).reshape(-1, 3)
    return rc, xyz, nrm


def write_flat(path, xyz, nrm):
    with open(path, "wb") as f:
        f.write(struct.pack("<QQ", len(xyz), len(nrm)))
        f.write(np.ascontiguousarray(xyz, np.float32).tobytes())
        f.write(np.ascontiguousarray(nrm, np.float32).tobytes())


@pytest.mark.parametrize("fmt", list(FORMATS))
@pytest.mark.parametrize("with_normals", [True, False])
def test_reads_reference_bytes_and_writes_them_back(tool, fix, tmp_path, fmt, with_normals):
    key = fmt if with_normals else fmt + "_no_normals"
    src = str(tmp_path / "ref.ply")
    open(src, "wb").write(fix[key].tobytes())
    rc, xyz, nrm = read_flat(tool, src, tmp_path)
    assert rc == 0
    want_n = fix["normals"] if with_normals else fix["normals"][:0]
    if fmt == "ascii":  # six decimals on disk
        assert np.allclose(xyz, fix["xyz"], atol=1e-6, rtol=1e-6) and len(nrm) == len(want_n)
        assert np.allclose(nrm, want_n, atol=1e-6, rtol=1e-6)
    else:
        assert np.array_equal(xyz, fix["xyz"]) and np.array_equal(nrm, want_n)
    # writer: same bytes as the reference writer for the same cloud
    flat, mine = str(tmp_path / "in.bin"), str(tmp_path / "mine.ply")
    write_flat(flat, fix["xyz"], want_n)
    subprocess.run([tool, "write", flat, mine, FORMATS[fmt]], check=True)
    assert open(mine, "rb").read() == fix[key].tobytes()
    # typed read -> typed write is the identity on the reference's bytes
    again = str(tmp_path / "again.ply")
    subprocess.run([tool, "copy", src, again, FORMATS[fmt]], check=True)
    assert open(again, "rb").read() == fix[key].tobytes()


def test_rejects_what_the_reference_rejects(tool, tmp_path):
    cases = {
        "not_ply.ply": b"plx\nformat ascii 1.0\nend_header\n",
        "bad_names.ply": b"ply\nformat ascii 1.0\nelement vertex 1\nproperty float x\n"
                         b"property float z\nproperty float y\nend_header\n0 0 0\n",
        "list_prop.ply": b"ply\nformat ascii 1.0\nelement vertex 1\nproperty list uchar int x\n"
                         b"property float y\nproperty float z\nend_header\n0 0 0\n",
        "truncated.ply": b"ply\nformat binary_little_endian 1.0\nelement vertex 4\n"
                         b"property float x\nproperty float y\nproperty float z\nend_header\n"
                         + b"\0" * 20,
    }
    for name, data in cases.items():
        p = str(tmp_path / name)
        open(p, "wb").write(data)
        rc, xyz, nrm = read_flat(tool, p, tmp_path)
        assert rc == 1 and len(xyz) == 0 and len(nrm) == 0, name
    rc, xyz, _ = read_flat(tool, str(tmp_path / "missing.ply"), tmp_path)
    assert rc == 1 and len(xyz) == 0


def test_comments_doubles_and_extra_elements(tool, tmp_path):
    pts = np.array([[1.5, -2.25, 3.0], [0.1, 0.2, 0.3]], np.float64)
    header = (b"ply\nformat binary_little_endian 1.0\ncomment made by hand\n"
              b"element vertex 2\nproperty double x\nproperty double y\nproperty double z\n"
              b"element face 0\nproperty list uchar int vertex_indices\nend_header\n")
    p = str(tmp_path / "d.ply")
    open(p, "wb").write(header + pts.tobytes())
    rc, xyz, nrm = read_flat(tool, p, tmp_path)
    assert rc == 0 and len(nrm) == 0
    assert np.array_equal(xyz, pts.astype(np.float32))


def test_reference_scans_when_mounted(tool, tmp_path):
    from oracle_lib import REFERENCE_DIR, RefPly, have_ref_ply

    data = os.path.join(REFERENCE_DIR, "examples", "data") if REFERENCE_DIR else None
    if data is None or not os.path.isdir(data):
        pytest.skip("the reference's example scans need PCP_REFERENCE (a reference checkout)")
    expected = {"stanford_bunny.ply": 35947, "detergent.ply": 20266, "spray.ply": 14851,
                "fandisk.ply": 6475}

    ref = RefPly() if have_ref_ply() else None
    for name, n in expected.items():
        rc, xyz, nrm = read_flat(tool, os.path.join(data, name), tmp_path)
        assert rc == 0 and xyz.shape == (n, 3) and np.isfinite(xyz).all(), name
        if ref is not None:
            rx, rn = ref.read(open(os.path.join(data, name), "rb").read())
            assert np.array_equal(rx, xyz) and len(rn) == len(nrm)
