"""Pins the CPU oracles (test infrastructure) before anything is compared against them.

* oracle/seg_oracle.c  vs  committed golden vectors produced by the UNMODIFIED reference
  (tests/golden/segmentator_golden.npz, scripts/make_golden.py, and tests/golden/reference_digests.json), which the
  reference itself (libref_segmentator.so, built by oracle/Makefile where the reference tree is present) is checked against.
* oracle/tsdf_oracle.c has nothing to be pinned against ("parity unpinned": the reference ships no TSDF
  source); it is checked for internal consistency and against the analytic geometry of the synthetic scene."""
import hashlib
import os

import numpy as np
import pytest

import oracle_bindings as ob
import reference_golden as rg
from scannet_b200 import synth
from scannet_b200._lib import TsdfParams

G = os.path.join(os.path.dirname(__file__), "golden")


def golden():
    return np.load(os.path.join(G, "segmentator_golden.npz"))


def test_seg_oracle_gates381_golden(built):
    xyz, tri = synth.read_ply(os.path.join(G, "gates381.ply"))
    g = golden()
    for k, m in [(0.01, 20), (0.001, 20), (0.0001, 20), (0.05, 5), (0.01, 1), (0.5, 100)]:
        assert (ob.oracle_segment(xyz, tri, k, m) == g[f"gates381_k{k}_m{m}"]).all()
    ids = ob.oracle_segment(xyz, tri)
    assert hashlib.sha256(",".join(map(str, ids.tolist())).encode()).hexdigest() == \
        "b57dfeed67ef8e452b78e6faf99c0b7c8892d1a838d40f4bd328e6c328e36cbf"          # BASELINE.md
    assert len(set(ids.tolist())) == 78


def test_seg_oracle_synthetic_golden(built):
    g = golden()
    for name, (x, t) in {"grid60x50_s2": synth.make_grid_mesh(60, 50, 2), "adv_s3": synth.make_adversarial_mesh(3),
                         "grid250x200_s1": synth.make_grid_mesh(250, 200, 1)}.items():
        assert bytes(g[f"{name}_xyz_sha"]) == hashlib.sha256(x.tobytes() + t.tobytes()).digest(), "generator drifted"
        assert (ob.oracle_segment(x, t) == g[name]).all(), name


def test_seg_oracle_sort_and_kruskal_golden(built):
    g = golden()
    e = g["graph_edges_in"].copy()
    ob.seg_oracle().oracle_seg_sort_edges(e.ctypes.data, len(e))
    assert e.tobytes() == g["graph_edges_sorted"].tobytes()          # libstdc++ std::sort tie order


@pytest.mark.parametrize("n,kind", [(1000, "ties"), (100000, "ties"), (65536, "organ"), (300000, "rand"), (17, "ties"), (16, "ties"), (200000, "few")])
def test_seg_oracle_sort_vs_reference_stdsort(built, n, kind):
    rng = np.random.default_rng(n)
    e = np.zeros(n, ob.EDGE_DTYPE)
    if kind == "ties":
        e["w"] = (rng.integers(0, 50, n) / 7.0).astype(np.float32)
    elif kind == "rand":
        e["w"] = rng.random(n).astype(np.float32)
    elif kind == "few":
        e["w"] = rng.integers(0, 3, n).astype(np.float32)
    else:
        e["w"] = np.concatenate([np.arange(n // 2), np.arange(n - n // 2)[::-1]]).astype(np.float32)
    e["a"] = np.arange(n); e["b"] = rng.integers(0, n, n)
    e2 = e.copy()
    ob.seg_oracle().oracle_seg_sort_edges(e2.ctypes.data, n)

    def ref():
        e1 = e.copy()
        ob.ref_segmentator().ref_segment_graph(n + 1, n, e1.ctypes.data, 0.5, None, None)
        return rg.digest(e1)

    assert rg.digest(e2) == rg.expect(f"stdsort_{kind}_{n}", "libref_segmentator.so", rg.digest(e), ref)


def test_seg_oracle_vs_reference_feature_mesh(built, tmp_path):
    x, t = synth.make_feature_mesh(120, 90, seed=4)
    p = tmp_path / "f.ply"; synth.write_ply(p, x, t)
    ref = rg.expect("feature_mesh_120x90_s4", "libref_segmentator.so", rg.digest(x, t), lambda: rg.digest(ob.ref_segment_file(p, len(x))))
    assert rg.digest(ob.oracle_segment(x, t)) == ref


def test_tsdf_oracle_geometry(built):
    """zero crossing of the fused sdf sits on the analytic surface: |sdf - true distance along the ray| small"""
    p = TsdfParams(); p.voxel_size = 0.004; p.trunc_base = 0.02; p.trunc_scale = 0.01; p.depth_min = 0.1; p.depth_max = 6.0
    p.max_integration_distance = 4.0; p.weight_sample = 1; p.weight_max = 255; p.width = 160; p.height = 120; p.depth_shift = 1000.0
    D, Cc, P, K = synth.make_frames(2, seed=1, width=160, height=120, loop_frames=400, with_color=True)
    o = ob.OracleTsdf(p, threads=4)
    assert o.integrate(D[0], Cc[0], P[0], K) == 0
    c1 = o.counters()
    assert o.integrate(D[1], Cc[1], np.full((4, 4), -np.inf, np.float32), K) == 1      # invalid pose skipped
    assert o.counters()["frames_skipped"] == 1 and o.counters()["total_updated"] == c1["total_updated"]
    xyz, vox = o.export()
    assert len(xyz) > 100 and (vox["w"] <= 1).all() and vox["w"].max() == 1
    upd = vox["w"] > 0
    assert np.abs(vox["sdf"][upd]).max() <= 0.02 + 0.01 * 6.0
    # voxels with |sdf| < trunc lie within one voxel diagonal of a room wall or sphere
    sc = synth.BoxRoomScene(seed=1, width=160, height=120)
    loc = np.stack(np.meshgrid(np.arange(8), np.arange(8), np.arange(8), indexing="ij"), -1).reshape(-1, 3)   # (lx,ly,lz), lz fastest
    lin = loc[:, 0] + 8 * loc[:, 1] + 64 * loc[:, 2]
    w = (xyz[:, None, :] * 8 + loc[None]) * 0.004
    near = np.zeros(vox["sdf"].shape, bool); near[:, lin] = True
    sel = upd & (np.abs(vox["sdf"]) < 0.004)
    pts = np.zeros(vox["sdf"].shape + (3,)); pts[:, lin] = w
    q = pts[sel]
    dwall = np.minimum.reduce([q[:, 0], q[:, 1], q[:, 2], sc.size[0] - q[:, 0], sc.size[1] - q[:, 1], sc.size[2] - q[:, 2]])
    dsph = np.minimum.reduce([np.abs(np.linalg.norm(q - c, axis=1) - r) for c, r in sc.spheres])
    assert (np.minimum(dwall, dsph) < 0.012).mean() > 0.99


def test_tsdf_spec_frozen(built):
    """the TSDF/marching-cubes oracle reproduces the committed hashes (scripts/make_tsdf_golden.py): guards this
    repo's own spec against drift — it is NOT a pin against the reference, which has no TSDF source"""
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("mk", os.path.join(ob.ROOT, "scripts", "make_tsdf_golden.py"))
    mk = importlib.util.module_from_spec(spec); spec.loader.exec_module(mk)
    with open(os.path.join(G, "tsdf_spec_golden.json")) as fh:
        gold = json.load(fh)
    for c in gold["cases"]:
        r = mk.run({k: c[k] for k in ("name", "wh", "frames", "seed", "loop", "noise", "drop", "inv", "color", "over")})
        for k, v in r.items():
            assert c[k] == v, (c["name"], k)
