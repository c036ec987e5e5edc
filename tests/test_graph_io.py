"""Graph files in the reference's formats (.el / .sg): our readers and writers against fixtures written by the
reference's own writer (tests/golden/make_io_fixtures.py) and, where the reference library is present, round trips
through its reader.  CPU-only except the final device load."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

from gms_b200 import io as gio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_read_reference_written_files(golden):
    rec = golden["graphs"]["triangles_3"]
    directed, off, nbr = gio.read_sg(os.path.join(GOLD, "triangles_3_undirected.sg"))
    assert not directed and off.tolist() == rec["off"] and nbr.tolist() == rec["nbr"]
    s, d = gio.read_el(os.path.join(GOLD, "triangles_3_undirected.el"))
    assert len(s) == len(rec["nbr"]) and d.tolist() == rec["nbr"]
    directed, off, nbr = gio.read_sg(os.path.join(GOLD, "triangles_3_directed.sg"))
    assert directed and off[-1] == 11 and nbr.tolist() == [1, 2, 2, 3, 3, 6, 7, 7, 8, 9, 9]
    directed, off, nbr = gio.read_sg(os.path.join(GOLD, "kronecker_8.sg"))
    assert sha(off) + sha(nbr) == golden["generated"]["kronecker-8"]["csr_sha"]


def test_writer_is_byte_identical_to_the_reference(tmp_path):
    for name in ("triangles_3_undirected.sg", "triangles_3_directed.sg", "kronecker_8.sg"):
        directed, off, nbr = gio.read_sg(os.path.join(GOLD, name))
        out = tmp_path / name
        gio.write_sg(str(out), off, nbr, directed)
        assert out.read_bytes() == open(os.path.join(GOLD, name), "rb").read(), name
    directed, off, nbr = gio.read_sg(os.path.join(GOLD, "triangles_3_undirected.sg"))
    out = tmp_path / "t.el"
    gio.write_el(str(out), off, nbr)
    assert out.read_text() == open(os.path.join(GOLD, "triangles_3_undirected.el")).read()


def test_truncated_file_is_rejected(tmp_path):
    data = open(os.path.join(GOLD, "kronecker_8.sg"), "rb").read()
    bad = tmp_path / "bad.sg"
    bad.write_bytes(data[:len(data) // 2])
    with pytest.raises(ValueError):
        gio.read_sg(str(bad))
    with pytest.raises(ValueError):
        gio.load_graph(str(tmp_path / "graph.mtx"))


def test_round_trip_through_the_reference_reader(ref_or_none, orc, reference_cases, tmp_path):
    """Files our writer makes, read back: the CSR must be the one the reference's reader builds from them (stored in
    oracle/reference_cases.py; the library itself as well where it is present)."""
    from oracle import reference_cases as rc
    assert rc.round_trip_record(orc, orc) == reference_cases["round_trip"]
    ref = ref_or_none
    if ref is None:
        return
    o = rc.round_trip_case(orc)
    off, nbr = o.csr()
    p = str(tmp_path / "g.sg")
    gio.write_sg(p, off, nbr, False)
    back = ref.load_file(p)
    boff, bnbr = back.csr()
    assert (boff == off).all() and (bnbr == nbr).all() and back.tc_total() == o.tc_total()
    # an .el file written by us, built by the reference's reader + builder
    q = str(tmp_path / "g.el")
    gio.write_el(q, off, nbr)
    back = ref.load_file(q, True)
    boff, bnbr = back.csr()
    assert (boff == off).all() and (bnbr == nbr).all()


def test_cpp_graph_io_compiles(gms):
    src = os.path.join(ROOT, "tests", "cpp", "graph_io_test.cpp")
    exe = os.path.join(ROOT, "build", "graph_io_test")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    lib = os.path.join(ROOT, "gms_b200", "lib")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), src, "-L" + lib, "-lgmsb",
                           "-Wl,-rpath," + lib, "-o", exe])


@pytest.mark.gpu
def test_load_graph_on_device(gms, golden, tmp_path):
    g = gio.load_graph(os.path.join(GOLD, "kronecker_8.sg"))
    assert g.tc_total() == golden["generated"]["kronecker-8"]["tc"]
    g = gio.load_graph(os.path.join(GOLD, "triangles_3_undirected.el"), symmetrize=True)
    assert g.tc_total() == 3 and g.tc_vertex2().tolist() == golden["graphs"]["triangles_3"]["vertex2"]
    exe = os.path.join(ROOT, "build", "graph_io_test")
    test_cpp_graph_io_compiles(gms)
    r = subprocess.run([exe, os.path.join(GOLD, "kronecker_8.sg"), os.path.join(GOLD, "triangles_3_directed.sg"),
                        str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert str(golden["generated"]["kronecker-8"]["tc"]) in r.stdout
    assert (tmp_path / "out.sg").read_bytes() == open(os.path.join(GOLD, "kronecker_8.sg"), "rb").read()
    assert (tmp_path / "dir.sg").read_bytes() == open(os.path.join(GOLD, "triangles_3_directed.sg"), "rb").read()
