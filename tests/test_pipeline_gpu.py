"""GPU: marching cubes parity, and the three CLIs end to end (.sens -> TSDF -> mesh -> segs.json)."""
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle_bindings as ob
import reference_golden as rg
from scannet_b200 import synth, tsdf

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "scannet_b200", "bin")
G = os.path.join(ROOT, "tests", "golden")


@pytest.mark.parametrize("wh,frames,color", [((96, 72), 4, True), ((160, 120), 6, False)])
def test_marching_cubes_matches_oracle(built, wh, frames, color):
    """identical vertex positions (bits), colours, triangle indices and order"""
    p = tsdf.default_params(width=wh[0], height=wh[1], max_blocks=1 << 15, hash_slots=1 << 17, batch_frames=3)
    D, Cc, P, K = synth.make_frames(frames, seed=7, width=wh[0], height=wh[1], loop_frames=400, noise_mm=1.0, drop=0.01)
    if not color:
        Cc = None
    vol = tsdf.TsdfVolume(p, device=0)
    vol.integrate_batch(D, Cc, P, K); vol.sync()
    gx, gc, gt = vol.extract_mesh()
    o = ob.OracleTsdf(p, threads=8)
    for i in range(frames):
        o.integrate(D[i], None if Cc is None else Cc[i], P[i], K)
    ox, oc, ot = o.extract_mesh()
    assert gx.shape == ox.shape and gt.shape == ot.shape and len(gt) > 1000
    assert gx.view(np.uint32).tobytes() == ox.view(np.uint32).tobytes()
    assert (gc == oc).all() and (gt == ot).all()
    # run twice: deterministic although heap indices are assigned by atomics
    gx2, gc2, gt2 = vol.extract_mesh()
    assert gx2.tobytes() == gx.tobytes() and (gt2 == gt).all()


def test_empty_volume_mesh(built):
    vol = tsdf.TsdfVolume(tsdf.default_params(width=32, height=24, max_blocks=64, hash_slots=256), device=0)
    x, c, t = vol.extract_mesh()
    assert len(x) == 0 and len(t) == 0


def segmentator_cli_digest(tool, d):
    """stdout and segs.json bytes of `tool` on a copy of gates381.ply in directory d (default and explicit parameters), then
    the usage text and status without arguments"""
    d.mkdir()
    shutil.copy(os.path.join(G, "gates381.ply"), d / "gates381.ply")
    parts = []
    for args, out in (((), "gates381.0.010000.segs.json"), (("0.05", "5"), "gates381.0.050000.segs.json")):
        o = subprocess.run([tool, str(d / "gates381.ply"), *args], capture_output=True, text=True)
        assert o.returncode == 0, o.stderr
        parts += [o.stdout.replace(str(d), "X"), (d / out).read_bytes().replace(str(d).encode(), b"X")]
    u = subprocess.run([tool], capture_output=True, text=True)
    assert u.returncode == 255
    return rg.digest(*parts, u.stdout)


def test_segmentator_cli_matches_reference_binary(built, tmp_path):
    """same stdout, same <base>.0.010000.segs.json bytes as the unmodified reference binary"""
    with open(os.path.join(G, "gates381.ply"), "rb") as fh:
        inputs = rg.digest(fh.read())
    ref = rg.expect("segmentator_cli_gates381", "segmentator_ref", inputs,
                    lambda: segmentator_cli_digest(os.path.join(ROOT, "oracle", "_ref", "segmentator_ref"), tmp_path / "b"))
    assert segmentator_cli_digest(os.path.join(BIN, "segmentator"), tmp_path / "a") == ref


def test_fuse_then_segment_end_to_end(built, tmp_path):
    """synthetic .sens (zlib depth, raw colour, one invalid pose) -> fuse -> _vh.ply -> segmentator -> segs.json"""
    D, Cc, P, K = synth.make_frames(24, seed=3, width=160, height=120, loop_frames=600, invalid_pose_every=11)
    sens = tmp_path / "scene.sens"
    synth.write_sens(str(sens), D, Cc, P, K, depth_comp=1, color_comp=0)
    params = tmp_path / "params.txt"
    params.write_text("s_SDFVoxelSize = 0.008f; // coarse for the test\ns_SDFTruncation = 0.04f;\ns_SDFTruncationScale = 0.01f;\ns_hashNumSDFBlocks = 60000;\n")
    r = subprocess.run([os.path.join(BIN, "fuse"), str(params), str(sens)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "integrated 22 frames (2 skipped" in r.stdout
    ply = tmp_path / "scene_vh.ply"
    assert ply.exists()
    xyz, tri = synth.read_ply(str(ply))
    assert len(xyz) > 5000 and len(tri) > 10000 and tri.max() < len(xyz)
    # vertices lie on the room / spheres
    sc = synth.BoxRoomScene(seed=3, width=160, height=120)
    q = xyz.astype(np.float64)
    dwall = np.minimum.reduce([q[:, 0], q[:, 1], q[:, 2], sc.size[0] - q[:, 0], sc.size[1] - q[:, 1], sc.size[2] - q[:, 2]])
    dsph = np.minimum.reduce([np.abs(np.linalg.norm(q - c, axis=1) - r_) for c, r_ in sc.spheres])
    assert (np.minimum(np.abs(dwall), dsph) < 0.02).mean() > 0.98
    r2 = subprocess.run([os.path.join(BIN, "segmentator"), str(ply)], capture_output=True, text=True)
    assert r2.returncode == 0, r2.stderr
    js = json.loads((tmp_path / "scene_vh.0.010000.segs.json").read_text())
    seg = np.array(js["segIndices"])
    assert len(seg) == len(xyz) and js["params"] == {"kThresh": 0.01, "segMinVerts": 20} and js["sceneId"] == "/scene_vh"
    # identical ids from the oracle on the same mesh
    assert (seg == ob.oracle_segment(xyz, tri)).all()
    assert 3 <= len(set(seg.tolist())) < len(xyz) // 20


def test_fuse_gpu_decode_writes_the_same_mesh(built, tmp_path):
    """`fuse` with the depth streams inflated on the GPU == `fuse` with the host decoder (same PLY bytes)."""
    D, Cc, P, K = synth.make_frames(40, seed=5, width=160, height=120, loop_frames=600, invalid_pose_every=13, noise_mm=1.0, drop=0.02)
    params = tmp_path / "params.txt"
    params.write_text("s_SDFVoxelSize = 0.008f;\ns_SDFTruncation = 0.04f;\ns_SDFTruncationScale = 0.01f;\ns_hashNumSDFBlocks = 60000;\n")
    out = {}
    for mode in ("host", "gpu"):
        d = tmp_path / mode; d.mkdir()
        synth.write_sens(str(d / "scene.sens"), D, Cc, P, K, depth_comp=1, color_comp=0)
        r = subprocess.run([os.path.join(BIN, "fuse"), str(params), str(d / "scene.sens")], capture_output=True, text=True,
                           env=dict(os.environ, SCN_FUSE_DECODE=mode))
        assert r.returncode == 0, r.stdout + r.stderr
        assert ("GPU inflate" in r.stdout) == (mode == "gpu")
        out[mode] = (d / "scene_vh.ply").read_bytes()
    assert out["host"] == out["gpu"]


def _jpeg_encoder(q=85):
    import cv2
    def enc(rgb):
        ok, buf = cv2.imencode(".jpg", rgb[:, :, ::-1], [int(cv2.IMWRITE_JPEG_QUALITY), q, int(cv2.IMWRITE_JPEG_SAMPLING_FACTOR), 0x221111])
        assert ok
        return buf.tobytes()
    return enc


def test_fuse_jpeg_colour_decoded_on_the_gpu_gives_the_host_decoders_mesh(built, tmp_path):
    """.sens with zlib depth + JPEG colour at a different resolution than depth: `fuse` with everything decoded in HBM (GPU
    inflate + GPU JPEG sampling only the registered pixels) writes the same coloured PLY as the host thread pool."""
    D, Cc, P, K = synth.make_frames(36, seed=7, width=160, height=120, loop_frames=500, invalid_pose_every=9, noise_mm=1.0)
    big = np.repeat(np.repeat(Cc, 2, axis=1), 2, axis=2)[:, :236, :318]                      # 318x236 colour for 160x120 depth
    Kc = K.copy(); Kc[0, 0] *= 318 / 160; Kc[1, 1] *= 236 / 120; Kc[0, 2] = (K[0, 2] + 0.5) * 318 / 160 - 0.5; Kc[1, 2] = (K[1, 2] + 0.5) * 236 / 120 - 0.5
    params = tmp_path / "params.txt"
    params.write_text("s_SDFVoxelSize = 0.008f;\ns_SDFTruncation = 0.04f;\ns_SDFTruncationScale = 0.01f;\ns_hashNumSDFBlocks = 60000;\n")
    out = {}
    for mode in ("host", "gpu"):
        d = tmp_path / mode; d.mkdir()
        synth.write_sens(str(d / "scene.sens"), D, big, P, K, K_color=Kc, depth_comp=1, color_comp=2, jpeg_encoder=_jpeg_encoder())
        r = subprocess.run([os.path.join(BIN, "fuse"), str(params), str(d / "scene.sens")], capture_output=True, text=True,
                           env=dict(os.environ, SCN_FUSE_DECODE=mode, SCN_FUSE_CHUNK="16"))
        assert r.returncode == 0, r.stdout + r.stderr
        assert ("GPU JPEG" in r.stdout) == (mode == "gpu")
        assert "integrated 32 frames (4 skipped" in r.stdout
        out[mode] = (d / "scene_vh.ply").read_bytes()
    assert out["host"] == out["gpu"]
    assert b"property uchar red" in out["gpu"][:400]


def test_fuse_many_scenes_library_driver(built, tmp_path):
    """scn_fuse_many: several scenes over the visible GPUs (one scene per GPU at a time); every report filled, meshes identical to
    the single-scene driver's"""
    from scannet_b200 import fuse as sfuse
    paths = []
    for i in range(3):
        D, Cc, P, K = synth.make_frames(20 + 4 * i, seed=20 + i, width=160, height=120, loop_frames=400)
        p = tmp_path / f"s{i}.sens"
        synth.write_sens(str(p), D, None, P, K, depth_comp=1, color_comp=0)
        paths.append(str(p))
    over = dict(voxel_size=0.008, trunc_base=0.04, max_blocks=60000, hash_slots=1 << 18)
    outs = [str(tmp_path / f"m{i}.ply") for i in range(3)]
    import torch
    devs = list(range(min(2, torch.cuda.device_count())))
    reps = sfuse.fuse_many(paths, outs, devices=devs, **over)
    assert [r["frames_integrated"] for r in reps] == [20, 24, 28] and all(r["status"] == 0 and r["mesh_faces"] > 1000 for r in reps)
    single = sfuse.fuse_scene(paths[1], str(tmp_path / "single.ply"), **over)
    assert single["mesh_vertices"] == reps[1]["mesh_vertices"]
    assert (tmp_path / "single.ply").read_bytes() == (tmp_path / "m1.ply").read_bytes()
    from scannet_b200 import ScnError
    with pytest.raises(ScnError):
        sfuse.fuse_many(paths + [str(tmp_path / "missing.sens")], None, devices=devs, **over)


def test_pooled_volume_is_reset_between_scenes_and_can_be_released(built, tmp_path):
    """Consecutive scenes of a process reuse the pooled volume (reset, not re-created): the second run of the same scene writes the
    same mesh bytes; a different scene in between leaves nothing behind; scn_release_cached_staging drops the pool."""
    from scannet_b200 import fuse as sfuse
    from scannet_b200._lib import lib
    paths = []
    for i in range(2):
        D, Cc, P, K = synth.make_frames(18 + 6 * i, seed=40 + i, width=160, height=120, loop_frames=400)
        p = tmp_path / f"s{i}.sens"
        synth.write_sens(str(p), D, None, P, K, depth_comp=1, color_comp=0)
        paths.append(str(p))
    over = dict(voxel_size=0.008, trunc_base=0.04, max_blocks=50000, hash_slots=1 << 18)
    assert lib().scn_release_cached_staging() == 0
    a = sfuse.fuse_scene(paths[0], str(tmp_path / "a.ply"), **over)
    b = sfuse.fuse_scene(paths[1], str(tmp_path / "b.ply"), **over)           # other scene, same layout: reuses a's volume
    c = sfuse.fuse_scene(paths[0], str(tmp_path / "c.ply"), **over)
    assert a["volume_reused"] == 0 and b["volume_reused"] == 1 and c["volume_reused"] == 1
    assert (tmp_path / "a.ply").read_bytes() == (tmp_path / "c.ply").read_bytes()
    assert a["blocks_allocated"] == c["blocks_allocated"] and a["voxels_updated"] == c["voxels_updated"]
    d = sfuse.fuse_scene(paths[0], None, **dict(over, max_blocks=40000))          # other layout: a new volume
    assert d["volume_reused"] == 0 and d["voxels_updated"] == a["voxels_updated"]
    assert lib().scn_release_cached_staging() == 0
    e = sfuse.fuse_scene(paths[0], None, **dict(over, max_blocks=40000))
    assert e["volume_reused"] == 0
