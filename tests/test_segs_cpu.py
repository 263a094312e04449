"""CPU: the segs.json consumer oracle (oracle/segs_oracle.c) pinned against the real mLib operators
(oracle/_ref/libref_mlib.so, compiled from the reference's external/mLib/include where it lies; their outputs are stored in
tests/golden/reference_digests.json), plus the segs.json reader (host code, no GPU needed)."""
import json

import numpy as np
import pytest

import oracle_bindings as ob
import reference_golden as rg
from scannet_b200 import segs, synth


def float_digest(a):
    """digest of the float32 bits, every NaN counted as the same value"""
    a = np.ascontiguousarray(a, np.float32)
    return rg.digest(np.where(np.isnan(a), np.float32(np.nan), a))


def test_area_matches_mlib(built):
    rng = np.random.default_rng(3)
    tris = rng.normal(size=(4000, 3, 3)).astype(np.float32)
    tris[:50, 2] = tris[:50, 0] + 2 * (tris[:50, 1] - tris[:50, 0])            # collinear -> the 1e-5 cosine guard
    tris[50:60, 1] = tris[50:60, 0]                                            # zero-length side -> NaN cosine
    o = ob.segs_oracle()
    a = np.array([o.oracle_tri_area_mlib(t[0].ctypes.data, t[1].ctypes.data, t[2].ctypes.data) for t in tris], np.float32)

    def ref():
        r = ob.ref_mlib()
        return float_digest(np.array([r.ref_tri_area(t[0].ctypes.data, t[1].ctypes.data, t[2].ctypes.data) for t in tris], np.float32))

    assert float_digest(a) == rg.expect("mlib_triangle_area", "libref_mlib.so", rg.digest(tris), ref)
    assert (a[:50] == 0).all() and np.isnan(a[50:60]).all()


@pytest.mark.parametrize("mesh", ["grid", "adversarial"])
def test_vertex_normals_match_mlib(built, mesh):
    xyz, tri = synth.make_feature_mesh(60, 50, 1) if mesh == "grid" else synth.make_adversarial_mesh(0)
    ref = rg.expect(f"mlib_vertex_normals_{mesh}", "libref_mlib.so", rg.digest(xyz, tri), lambda: float_digest(ob.ref_vertex_normals_mlib(xyz, tri)))
    assert float_digest(ob.oracle_vertex_normals_mlib(xyz, tri)) == ref


def test_aggregate_oracle_matches_python_dicts(built):
    """Segmentation.h:68-75 builds map<segId, vector<vertId>> by push_back in vertex order."""
    rng = np.random.default_rng(0)
    seg = rng.integers(0, 40, 1000).astype(np.uint32) * 7
    r = ob.oracle_segs_aggregate(seg)
    d = {}
    for i, s in enumerate(seg):
        d.setdefault(int(s), []).append(i)
    assert list(r["seg_ids"]) == sorted(d)
    for k, s in enumerate(r["seg_ids"]):
        assert list(r["vert_ids"][int(r["offsets"][k]):int(r["offsets"][k + 1])]) == d[int(s)]


def test_segs_json_reader(tmp_path, built):
    p = tmp_path / "a.segs.json"
    p.write_text('{"params":{"kThresh":0.01,"segMinVerts":20},"sceneId":"/gates381","segIndices":[5,5,"7",null,0,4294967295,12]}')
    r = segs.load(str(p))
    assert list(r["segIndices"]) == [5, 5, 7, 0xFFFFFFFF, 0, 0xFFFFFFFF, 12]
    assert abs(r["kThresh"] - 0.01) < 1e-9 and r["segMinVerts"] == 20 and r["sceneId"] == "/gates381"
    # the layout Segmentation::saveToFile writes (Segmentation.h:90-106): multi-line, extra params, other member order
    q = tmp_path / "b.segs.json"
    q.write_text('{\n"params": {"kThresh": "0.5", "minPoints": 3, "nested": {"a": [1, {"b": "]"}]}},\n"sceneId": "scene0000_00",\n"extra": [1, 2, {"x": null}],\n"segIndices": [1,2,3]\n}\n')
    r = segs.load(str(q))
    assert list(r["segIndices"]) == [1, 2, 3] and r["kThresh"] == 0.5 and r["segMinVerts"] == 0 and r["sceneId"] == "scene0000_00"
    e = tmp_path / "empty.json"; e.write_text('{"segIndices":[]}')
    assert len(segs.load(str(e))["segIndices"]) == 0


def test_segs_json_reader_errors(tmp_path, built):
    from scannet_b200._lib import ScnError
    with pytest.raises(ScnError, match="failed to open"):
        segs.load(str(tmp_path / "missing.json"))
    bad = tmp_path / "bad.json"; bad.write_text('{"segIndices":[1,2,')
    with pytest.raises(ScnError, match="Parse error"):
        segs.load(str(bad))
    none = tmp_path / "none.json"; none.write_text('{"sceneId":"x"}')
    with pytest.raises(ScnError, match="segIndices"):
        segs.load(str(none))


def test_segmentator_output_round_trips_through_reader(tmp_path, built):
    """what scn_write_segs_json writes (segmentator.cpp:253-266 layout) is what the reader returns"""
    import ctypes as C
    from scannet_b200._lib import check, lib
    ids = np.array([3, 3, 9, 0, 2147483647], np.int32)
    p = tmp_path / "x.0.010000.segs.json"
    check(lib().scn_write_segs_json(str(p).encode(), b"/x", C.c_float(0.01), C.c_int32(20), ids.ctypes.data_as(C.c_void_p), C.c_uint64(len(ids))))
    assert json.loads(p.read_text())["segIndices"] == ids.tolist()
    r = segs.load(str(p))
    assert r["segIndices"].tolist() == ids.tolist() and r["sceneId"] == "/x" and r["segMinVerts"] == 20
