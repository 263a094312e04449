"""GPU: the scene driver (scn_fuse_scene) in both decode modes.  Every decoder path writes the same mesh, a frame that fails to
decode fails the scene with its own status code, and a pose-less frame is never decoded."""
import os
import struct

import numpy as np
import pytest

from scannet_b200 import ScnError, fuse, synth

pytestmark = pytest.mark.gpu
SCN_ERR_ARG, SCN_ERR_IO, SCN_ERR_FORMAT = -1, -3, -4
OVER = dict(voxel_size=0.008, trunc_base=0.04, trunc_scale=0.01, max_blocks=60000, hash_slots=1 << 18)


def scene(n_frames):
    """160x120 frames along a camera loop; every 7th pose is invalid"""
    return synth.make_frames(n_frames, seed=5, width=160, height=120, loop_frames=600, invalid_pose_every=7, noise_mm=1.0, drop=0.02)


def fuse_both_modes(sens, tmp_path, tag):
    """{mode: (report, PLY bytes)}"""
    out = {}
    for mode in ("gpu", "host"):
        ply = tmp_path / f"{tag}_{mode}.ply"
        rep = fuse.fuse_scene(str(sens), str(ply), decode_mode=mode, **OVER)
        assert rep["gpu_decode"] == (mode == "gpu")
        out[mode] = (rep, ply.read_bytes())
    return out


def test_every_decoder_path_writes_the_same_mesh(built, tmp_path, monkeypatch):
    """zlib and raw depth, each through the GPU decoders (16-frame chunks) and the host decoders (several chunks as well)"""
    monkeypatch.setenv("SCN_FUSE_CHUNK", "16")
    D, Cc, P, K = scene(max(32, 2 * min(64, os.cpu_count() or 1)) + 40)        # more frames than one host-mode chunk
    n_poseless = int((P[:, 0, 0] == -np.inf).sum())
    runs = []
    for depth_comp in (1, 0):
        sens = tmp_path / f"depth{depth_comp}.sens"
        synth.write_sens(str(sens), D, Cc, P, K, depth_comp=depth_comp, color_comp=0)
        runs += fuse_both_modes(sens, tmp_path, f"depth{depth_comp}").values()
    meshes = [ply for _, ply in runs]
    assert all(m == meshes[0] for m in meshes) and b"property uchar red" in meshes[0][:400]
    for rep, _ in runs:
        assert rep["frames_integrated"] == len(D) - n_poseless
        assert rep["frames_skipped"] == rep["frames_skipped_pose"] == n_poseless


def test_png_colour_gives_the_raw_colour_mesh(built, tmp_path, monkeypatch):
    """PNG colour is decoded by the host pool in both modes (and uploaded once per chunk in GPU mode); PNG is lossless"""
    import cv2
    monkeypatch.setenv("SCN_FUSE_CHUNK", "16")
    D, Cc, P, K = scene(48)
    png, raw = tmp_path / "png.sens", tmp_path / "raw.sens"
    synth.write_sens(str(png), D, Cc, P, K, depth_comp=1, color_comp=1, jpeg_encoder=lambda rgb: cv2.imencode(".png", rgb[:, :, ::-1])[1].tobytes())
    synth.write_sens(str(raw), D, Cc, P, K, depth_comp=1, color_comp=0)
    out = fuse_both_modes(png, tmp_path, "png")
    assert out["gpu"][1] == out["host"][1]
    assert out["gpu"][1] == fuse_both_modes(raw, tmp_path, "raw")["gpu"][1]


def depth_payloads(path):
    """(offset, bytes) of every frame's depth payload in a .sens file (layout: scannet_b200.synth.write_sens)"""
    buf = open(path, "rb").read()
    o = 4 + 8 + struct.unpack_from("<Q", buf, 4)[0] + 4 * 64 + 8 + 16 + 4
    n = struct.unpack_from("<Q", buf, o)[0]
    o += 8
    out = []
    for _ in range(n):
        cb, db = struct.unpack_from("<QQ", buf, o + 64 + 16)
        out.append((o + 64 + 32 + cb, db))
        o += 64 + 32 + cb + db
    return out


def with_corrupt_depth(src, dst, frame):
    """a copy of `src` whose frame `frame` has a zlib depth stream with a reserved deflate block type"""
    buf = bytearray(open(src, "rb").read())
    off, n = depth_payloads(src)[frame]
    buf[off:off + n] = b"\x78\x9c" + b"\xff" * (n - 2)
    open(dst, "wb").write(bytes(buf))


def test_corrupt_depth_payload(built, tmp_path, monkeypatch):
    """on a frame with a pose it fails the scene with SCN_ERR_FORMAT and the file's name, and the next scene gets a new volume; on
    a pose-less frame it is never decoded"""
    monkeypatch.setenv("SCN_FUSE_CHUNK", "16")
    D, Cc, P, K = scene(48)
    good = tmp_path / "good.sens"
    synth.write_sens(str(good), D, Cc, P, K, depth_comp=1, color_comp=0)
    posed = [i for i in range(len(P)) if P[i, 0, 0] != -np.inf]
    poseless = [i for i in range(len(P)) if P[i, 0, 0] == -np.inf]
    bad = tmp_path / "bad.sens"
    with_corrupt_depth(good, bad, posed[20])
    for mode in ("gpu", "host"):
        with pytest.raises(ScnError) as e:
            fuse.fuse_scene(str(bad), str(tmp_path / "bad.ply"), decode_mode=mode, **OVER)
        assert e.value.code == SCN_ERR_FORMAT and str(bad) in str(e.value)
        assert fuse.fuse_scene(str(good), None, decode_mode=mode, **OVER)["volume_reused"] == 0
    skip = tmp_path / "skip.sens"
    with_corrupt_depth(good, skip, poseless[1])
    clean = fuse_both_modes(good, tmp_path, "clean")["host"][1]
    assert all(ply == clean for _, ply in fuse_both_modes(skip, tmp_path, "skip").values())


def test_failures_keep_their_status_code(built, tmp_path):
    D, Cc, P, K = scene(12)
    sens = tmp_path / "scene.sens"
    synth.write_sens(str(sens), D, Cc, P, K, depth_comp=1, color_comp=0)
    with pytest.raises(ScnError) as e:
        fuse.fuse_scene(str(sens), str(tmp_path / "missing" / "scene.ply"), **OVER)
    assert e.value.code == SCN_ERR_IO and str(sens) in str(e.value)
    with pytest.raises(ScnError) as e:
        fuse.fuse_scene(str(sens), None, **dict(OVER, voxel_size=0.0))
    assert e.value.code == SCN_ERR_ARG and str(sens) in str(e.value)
