#!/usr/bin/env python
"""Regenerates tests/golden/* by running the UNMODIFIED reference (oracle/_ref, built from
/root/reference by oracle/Makefile) in this container.  The GPU box has no /root/reference, so the
vectors are committed.  Usage: python scripts/make_golden.py"""
import hashlib
import os
import shutil
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_bindings as ob  # noqa: E402
from scannet_b200 import synth  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")
REF_MESH = "/root/reference/external/mLib/test/testD3D11/scans/gates381.ply"


def sha(ids):
    return hashlib.sha256(",".join(map(str, ids.tolist())).encode()).hexdigest()


def main():
    os.makedirs(G, exist_ok=True)
    # the only mesh fixture in the reference tree (mLib test data, VCGLIB binary PLY; data, not source)
    shutil.copyfile(REF_MESH, os.path.join(G, "gates381.ply"))
    os.chmod(os.path.join(G, "gates381.ply"), 0o644)
    xyz, tri = synth.read_ply(REF_MESH)
    out = {}
    for k, m in [(0.01, 20), (0.001, 20), (0.0001, 20), (0.05, 5), (0.01, 1), (0.5, 100)]:
        ids = ob.ref_segment_file(REF_MESH, len(xyz), k, m)
        out[f"gates381_k{k}_m{m}"] = ids
        print("gates381", k, m, len(set(ids.tolist())), sha(ids))
    assert sha(out["gates381_k0.01_m20"]) == "b57dfeed67ef8e452b78e6faf99c0b7c8892d1a838d40f4bd328e6c328e36cbf"  # BASELINE.md
    # reference segment_graph (std::sort + Kruskal) on a tie-heavy synthetic edge list
    rng = np.random.default_rng(7)
    n = 50000
    e = np.zeros(n, ob.EDGE_DTYPE)
    e["w"] = (rng.integers(0, 40, n) / 13.0).astype(np.float32); e["a"] = rng.integers(0, 5000, n); e["b"] = rng.integers(0, 5000, n)
    es = e.copy(); roots = np.zeros(5000, np.int32); sizes = np.zeros(5000, np.int32)
    ob.ref_segmentator().ref_segment_graph(5000, n, es.ctypes.data, 0.3, roots.ctypes.data, sizes.ctypes.data)
    out["graph_edges_in"] = e; out["graph_edges_sorted"] = es; out["graph_roots"] = roots; out["graph_sizes"] = sizes
    # synthetic + adversarial meshes through the reference CLI path (file -> ids)
    for name, (x, t) in {"grid60x50_s2": synth.make_grid_mesh(60, 50, 2), "adv_s3": synth.make_adversarial_mesh(3),
                         "grid250x200_s1": synth.make_grid_mesh(250, 200, 1)}.items():
        p = f"/tmp/_golden_{name}.ply"; synth.write_ply(p, x, t)
        ids = ob.ref_segment_file(p, len(x))
        out[f"{name}_xyz_sha"] = np.frombuffer(hashlib.sha256(x.tobytes() + t.tobytes()).digest(), np.uint8)
        out[name] = ids
        print(name, len(x), len(set(ids.tolist())), sha(ids))
    np.savez_compressed(os.path.join(G, "segmentator_golden.npz"), **out)
    print("wrote", os.path.join(G, "segmentator_golden.npz"))


def fixtures(ref_root):
    """Data files of the reference tree the tests read: the two ScanNet reconstruction parameter files, and the first
    1000 vertices of the OBJ copy of gates381 with the faces among them (the whole file is 890 kB)."""
    for name in ("zParametersScanNet.txt", "zParametersBundlingScanNet.txt"):
        shutil.copyfile(os.path.join(ref_root, "Server", "tools", "recons", name), os.path.join(G, name))
        os.chmod(os.path.join(G, name), 0o644)
    keep, nv, lines = 1000, 0, []
    with open(os.path.join(ref_root, "external", "mLib", "test", "testD3D11", "scans", "gates381.obj")) as fh:
        for ln in fh:
            if ln.startswith("v "):
                nv += 1
                if nv > keep:
                    continue
            elif ln.startswith("vn "):
                if nv >= keep:
                    continue
            elif ln.startswith("f ") and max(int(x.split("/")[0]) for x in ln.split()[1:]) > keep:
                continue
            lines.append(ln)
    with open(os.path.join(G, "gates381_head1000.obj"), "w") as fh:
        fh.writelines(lines)


if __name__ == "__main__":
    if sys.argv[1:2] == ["fixtures"]:               # python scripts/make_golden.py fixtures <reference tree>
        fixtures(sys.argv[2])
    else:
        main()
