"""Mesh loaders + segs.json writer (host logic, no GPU): scn_mesh_load must hand the kernels exactly the
arrays the reference's tinyply / tinyobjloader paths produce (segmentator.cpp:130-172)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from scannet_b200 import synth
from scannet_b200._lib import check, lib

G = os.path.join(os.path.dirname(__file__), "golden")


def mesh_load(path):
    L = lib()
    xyz = C.POINTER(C.c_float)(); tri = C.POINTER(C.c_uint32)(); nv = C.c_uint64(); nf = C.c_uint64()
    check(L.scn_mesh_load(str(path).encode(), C.byref(xyz), C.byref(nv), C.byref(tri), C.byref(nf)))
    a = np.ctypeslib.as_array(xyz, (nv.value * 3,)).copy().reshape(-1, 3) if nv.value else np.zeros((0, 3), np.float32)
    t = np.ctypeslib.as_array(tri, (nf.value * 3,)).copy().reshape(-1, 3) if nf.value else np.zeros((0, 3), np.uint32)
    L.scn_free(xyz); L.scn_free(tri)
    return a, t


def test_ply_binary_le_matches_fixture(built):
    xyz, tri = mesh_load(os.path.join(G, "gates381.ply"))
    rx, rt = synth.read_ply(os.path.join(G, "gates381.ply"))
    assert xyz.shape == (5860, 3) and tri.shape == (10197, 3)
    assert xyz.tobytes() == rx.tobytes() and (tri == rt).all()


@pytest.mark.parametrize("fmt", ["ascii", "binary_big_endian", "binary_little_endian"])
def test_ply_variants(tmp_path, built, fmt):
    """extra properties before/after x,y,z, an extra element, 'vertex_index' naming, uint indices"""
    xyz, tri = synth.make_grid_mesh(9, 7, seed=1)
    p = tmp_path / "m.ply"
    V, F = len(xyz), len(tri)
    hdr = f"ply\nformat {fmt} 1.0\ncomment test\nelement vertex {V}\nproperty uchar flag\nproperty float x\nproperty float y\nproperty float z\n" \
          f"property double q\nelement edge 2\nproperty int a\nproperty list uchar short lst\nelement face {F}\nproperty list uchar uint vertex_index\nproperty uchar mat\nend_header\n"
    bo = ">" if fmt == "binary_big_endian" else "<"
    with open(p, "wb") as f:
        f.write(hdr.encode())
        if fmt == "ascii":
            for v in xyz:
                f.write(f"7 {float(v[0])!r} {float(v[1])!r} {float(v[2])!r} 0.5\n".encode())
            f.write(b"1 2 5 6\n2 0\n")
            for t in tri:
                f.write(f"3 {t[0]} {t[1]} {t[2]} 9\n".encode())
        else:
            v = np.zeros(V, dtype=[("flag", "u1"), ("x", bo + "f4"), ("y", bo + "f4"), ("z", bo + "f4"), ("q", bo + "f8")])
            v["x"], v["y"], v["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
            f.write(v.tobytes())
            f.write(np.array([1], bo + "i4").tobytes() + bytes([2]) + np.array([5, 6], bo + "i2").tobytes())
            f.write(np.array([2], bo + "i4").tobytes() + bytes([0]))
            fa = np.zeros(F, dtype=[("n", "u1"), ("i", bo + "u4", (3,)), ("mat", "u1")]); fa["n"] = 3; fa["i"] = tri; fa["mat"] = 9
            f.write(fa.tobytes())
    a, t = mesh_load(p)
    assert (t == tri).all()
    if fmt == "ascii":
        assert np.array_equal(a, xyz)      # repr() round-trips float32 exactly through the istream >> float path
    else:
        assert a.tobytes() == xyz.tobytes()


def test_obj_loader_semantics(tmp_path, built):
    """first shape only, original vertices, relative indices, v/vt/vn triples, CRLF, the decimal parser"""
    p = tmp_path / "m.obj"
    p.write_bytes(b"# c\r\nv 0.1 0.2 0.3\r\nv 1e-2 -2.5E1 +3\nv 0.30000001192092896 7 8 0.5 0.5 0.5\nv 1 1\nvn 0 0 1\nvt 0 0\n"
                  b"o first\nf 1/1/1 2//1 3\nf -1 -2 -3\ng second\nf 1 2 3\n")
    xyz, tri = mesh_load(p)
    assert xyz.shape == (4, 3) and tri.tolist() == [[0, 1, 2], [3, 2, 1]]
    assert xyz[3].tolist() == [1.0, 1.0, 0.0]
    # tinyobj's parser accumulates decimals in double with a power table: 0.1 -> 1*0.1, 0.2, 0.3 are exact here;
    # 1e-2 = ldexp(1 * 5^-2, -2)
    assert xyz[1, 0] == np.float32(np.ldexp(1.0 * 5.0 ** -2, -2)) and xyz[1, 1] == np.float32(-250.0 / 10)


def test_obj_matches_reference_on_gates381(tmp_path, built):
    """the first 1000 vertices of the reference's gates381.obj (scripts/make_golden.py) with the faces among them"""
    import oracle_bindings as ob
    import reference_golden as rg
    src = os.path.join(G, "gates381_head1000.obj")
    xyz, tri = mesh_load(src)
    assert xyz.shape == (1000, 3) and len(tri) > 1000
    with open(src, "rb") as fh:
        inputs = rg.digest(fh.read())
    ref_ids = rg.expect("gates381_head1000_obj", "libref_segmentator.so", inputs, lambda: rg.digest(ob.ref_segment_file(src, len(xyz))))
    ours = ob.oracle_segment(xyz, tri)          # same arrays -> same ids only if the loader parsed every float like tinyobj
    assert rg.digest(ours) == ref_ids


def test_segs_json_bytes(tmp_path, built):
    seg = np.array([5, 5, 0, 123456, 7], np.int32)
    p = tmp_path / "x.segs.json"
    check(lib().scn_write_segs_json(str(p).encode(), b"/scene0000_00_vh_clean_2", C.c_float(0.01), C.c_int32(20),
                                    seg.ctypes.data_as(C.c_void_p), C.c_uint64(len(seg))))
    txt = p.read_text()
    assert txt == '{"params":{"kThresh":0.01,"segMinVerts":20},"sceneId":"/scene0000_00_vh_clean_2","segIndices":[5,5,0,123456,7]}'
    assert json.loads(txt)["segIndices"] == seg.tolist()


def test_unsupported_inputs_are_errors(tmp_path, built):
    from scannet_b200 import ScnError
    p = tmp_path / "quad.ply"
    p.write_bytes(b"ply\nformat ascii 1.0\nelement vertex 4\nproperty float x\nproperty float y\nproperty float z\nelement face 1\n"
                  b"property list uchar int vertex_indices\nend_header\n0 0 0\n1 0 0\n1 1 0\n0 1 0\n4 0 1 2 3\n")
    with pytest.raises(ScnError):
        mesh_load(p)
    q = tmp_path / "junk.ply"; q.write_bytes(b"ply\nformat ascii 1.0\nbogus line\nend_header\n")
    with pytest.raises(ScnError):
        mesh_load(q)
    with pytest.raises(ScnError):
        mesh_load(tmp_path / "missing.ply")


def test_absurd_element_counts_are_errors_not_exceptions(tmp_path, built):
    """ADVICE r01: `element vertex 999999999999999999` used to throw std::length_error through the C ABI (process abort)."""
    import ctypes as C
    from scannet_b200._lib import lib
    for fmt, body in (("binary_little_endian", b"\x00" * 64), ("ascii", b"0 0 0\n")):
        p = tmp_path / f"huge_{fmt}.ply"
        p.write_bytes(("ply\nformat %s 1.0\nelement vertex 999999999999999999\nproperty float x\nproperty float y\nproperty float z\n"
                       "element face 0\nproperty list uchar int vertex_indices\nend_header\n" % fmt).encode() + body)
        px = C.POINTER(C.c_float)(); pt = C.POINTER(C.c_uint32)(); nv = C.c_uint64(); nf = C.c_uint64()
        rc = lib().scn_mesh_load(str(p).encode(), C.byref(px), C.byref(nv), C.byref(pt), C.byref(nf))
        assert rc != 0


def test_segs_json_integer_formatting_matches_printf(tmp_path, built):
    """The writer formats the ids itself (no snprintf): same bytes as "%d" for every sign and width."""
    import ctypes as C
    import json
    from scannet_b200._lib import lib
    rng = np.random.default_rng(3)
    ids = np.concatenate([np.array([0, 1, 9, 10, 99, 100, -1, -10, 2**31 - 1, -2**31, 123456789], np.int64),
                          rng.integers(-2**31, 2**31 - 1, 5000), rng.integers(0, 50000, 5000)]).astype(np.int32)
    p = str(tmp_path / "x.segs.json")
    assert lib().scn_write_segs_json(p.encode(), b"scene", C.c_float(0.01), C.c_int32(20), ids.ctypes.data_as(C.c_void_p), C.c_uint64(len(ids))) == 0
    txt = open(p).read()
    body = txt[txt.index('"segIndices":[') + len('"segIndices":['):-2]
    assert body == ",".join("%d" % int(v) for v in ids)
    assert json.loads(txt)["segIndices"] == [int(v) for v in ids]


@pytest.mark.parametrize("nv,with_rgb", [(50, True), (50, False), (120000, True), (120000, False)])
def test_ply_writer_bytes_small_and_mapped_paths(tmp_path, built, nv, with_rgb):
    """scn_mesh_save_ply: the buffered path (small files) and the mapped multi-threaded path (> 1 MB) write the same VCGLIB-layout
    bytes: header, 16-byte vertices (xyz + rgba, alpha 255, white without colour), 13-byte triangle records."""
    import ctypes as C
    from scannet_b200._lib import lib
    rng = np.random.default_rng(nv)
    xyz = rng.standard_normal((nv, 3)).astype(np.float32)
    rgb = rng.integers(0, 256, (nv, 3)).astype(np.uint8)
    tri = rng.integers(0, nv, (2 * nv, 3)).astype(np.uint32)
    p = str(tmp_path / "m.ply")
    rc = lib().scn_mesh_save_ply(p.encode(), xyz.ctypes.data_as(C.c_void_p), rgb.ctypes.data_as(C.c_void_p) if with_rgb else None, C.c_uint64(nv),
                                 tri.ctypes.data_as(C.c_void_p), C.c_uint64(len(tri)))
    assert rc == 0
    head = ("ply\nformat binary_little_endian 1.0\ncomment VCGLIB generated\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n"
            "property uchar red\nproperty uchar green\nproperty uchar blue\nproperty uchar alpha\nelement face %d\nproperty list uchar int vertex_indices\nend_header\n"
            % (nv, len(tri))).encode()
    v = np.zeros((nv, 16), np.uint8)
    v[:, :12] = xyz.view(np.uint8).reshape(nv, 12)
    v[:, 12:15] = rgb if with_rgb else 255
    v[:, 15] = 255
    f = np.zeros((len(tri), 13), np.uint8)
    f[:, 0] = 3
    f[:, 1:] = tri.view(np.uint8).reshape(len(tri), 12)
    assert open(p, "rb").read() == head + v.tobytes() + f.tobytes()
