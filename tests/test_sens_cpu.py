"""SensReader host logic (no GPU): `.sens` v4 container, depth/colour decode, writer, saveToImages —
byte-exact against the UNMODIFIED reference ml::SensorData (oracle/_ref/libref_sens.so, sens_ref), through the outputs of it
stored in tests/golden/reference_digests.json (reference_golden.py)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import reference_golden as rg
from scannet_b200 import synth
from scannet_b200.sens import SensFile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref_sens.so")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "sens_ref")


def ref_lib():
    L = C.CDLL(REF_SO)
    L.ref_sens_open.restype = C.c_void_p; L.ref_sens_open.argtypes = [C.c_char_p]
    L.ref_sens_close.argtypes = [C.c_void_p]
    L.ref_sens_info.argtypes = [C.c_void_p] * 7
    L.ref_sens_frame_meta.argtypes = [C.c_void_p, C.c_uint64] + [C.c_void_p] * 5
    L.ref_sens_depth.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    L.ref_sens_color.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    return L


def file_digest(p):
    with open(p, "rb") as fh:
        return rg.digest(fh.read())


def ref_colour(p, W, H, n=1):
    """digest of the reference's colour decode of the first n frames of the .sens file p (each must decode)"""
    L = ref_lib(); r = L.ref_sens_open(p.encode()); assert r
    out = []
    for i in range(n):
        rc = np.zeros((H, W, 3), np.uint8); assert L.ref_sens_color(r, i, rc.ctypes.data) == 0
        out.append(rc)
    L.ref_sens_close(r)
    return rg.digest(*out)


def jpeg_bytes(rgb, quality=85, subsample=None):
    import cv2
    params = [int(cv2.IMWRITE_JPEG_QUALITY), quality]
    if subsample is not None:
        params += [int(cv2.IMWRITE_JPEG_SAMPLING_FACTOR), subsample]
    ok, buf = cv2.imencode(".jpg", rgb[:, :, ::-1], params)
    assert ok
    return buf.tobytes()


@pytest.fixture(scope="module")
def stream(tmp_path_factory, built):
    d = tmp_path_factory.mktemp("sens")
    D, Cc, P, K = synth.make_frames(5, seed=2, width=160, height=120, loop_frames=50, noise_mm=2.0, drop=0.05, invalid_pose_every=4)
    rng = np.random.default_rng(0)
    Cc = np.clip(Cc.astype(np.int32) + rng.integers(-20, 20, Cc.shape), 0, 255).astype(np.uint8)   # texture for the JPEG path
    p = str(d / "synth.sens")
    synth.write_sens(p, D, Cc, P, K, depth_comp=1, color_comp=2, jpeg_encoder=jpeg_bytes)
    return p, D, Cc, P, K


def header_digest(dims, depth_shift, comp, n_frames, mats, frames):
    parts = [np.array(dims, np.uint32), np.float32(depth_shift), np.array(comp, np.int32), np.uint64(n_frames), np.array(mats, np.float32)]
    for T, meta, depth, color in frames:
        parts += [np.asarray(T, np.float32).reshape(16), np.array(meta, np.uint64), np.asarray(depth, np.uint16), np.asarray(color, np.uint8)]
    return rg.digest(*parts)


def test_header_and_frames_match_reference(stream):
    p, D, Cc, P, K = stream
    s = SensFile(p)
    i = s.info
    assert i.n_frames == 5
    frames = []
    for f in range(5):
        T2, tc, td, cb, db = s.frame_meta(f)
        assert (s.depth(f) == D[f]).all()
        frames.append((T2, (tc, td, cb, db), s.depth(f), s.color(f)))
    ours = header_digest([i.color_width, i.color_height, i.depth_width, i.depth_height], i.depth_shift, [i.color_compression, i.depth_compression],
                         i.n_frames, list(i.color_intrinsic) + list(i.color_extrinsic) + list(i.depth_intrinsic) + list(i.depth_extrinsic), frames)
    s.close()

    def ref():
        L = ref_lib(); r = L.ref_sens_open(p.encode())
        assert r
        dims = (C.c_uint32 * 4)(); ds = C.c_float(); comp = (C.c_int32 * 2)(); nf = C.c_uint64(); ni = C.c_uint64(); mats = (C.c_float * 64)()
        L.ref_sens_info(r, dims, C.byref(ds), comp, C.byref(nf), C.byref(ni), mats)
        rframes = []
        for f in range(5):
            T = np.zeros(16, np.float32); a = C.c_uint64(); b = C.c_uint64(); c = C.c_uint64(); d = C.c_uint64()
            L.ref_sens_frame_meta(r, f, T.ctypes.data, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
            rd = np.zeros((120, 160), np.uint16); assert L.ref_sens_depth(r, f, rd.ctypes.data) == 0
            assert (rd == D[f]).all()
            rc = np.zeros((120, 160, 3), np.uint8); assert L.ref_sens_color(r, f, rc.ctypes.data) == 0
            rframes.append((T, (a.value, b.value, c.value, d.value), rd, rc))
        L.ref_sens_close(r)
        return header_digest(list(dims), ds.value, list(comp), nf.value, list(mats), rframes)

    assert ours == rg.expect("sens_header_and_frames", "libref_sens.so", file_digest(p), ref), \
        "header, frame metadata, depth or JPEG decode (stb_image) differs from the reference"


@pytest.mark.parametrize("sub,wh", [(0x111111, (67, 45)), (0x211111, (66, 47)), (0x221111, (70, 33)), (0x121111, (64, 48)), (0x411111, (72, 40))])
def test_jpeg_subsampling_modes_match_stb(tmp_path, built, sub, wh):
    """4:4:4, 4:2:2, 4:2:0, 4:4:0, 4:1:1 chroma layouts at non-MCU-aligned sizes."""
    W, H = wh
    rng = np.random.default_rng(sub)
    yy, xx = np.mgrid[0:H, 0:W]
    img = np.stack([(xx * 5 + yy) % 256, (yy * 7) % 256, (xx * yy) % 256], -1).astype(np.uint8)
    img = np.clip(img.astype(int) + rng.integers(-30, 30, img.shape), 0, 255).astype(np.uint8)
    D = np.full((1, 8, 8), 1000, np.uint16); P = np.eye(4, dtype=np.float32)[None]
    p = str(tmp_path / "j.sens")
    synth.write_sens(p, D, img[None], P, np.eye(4, dtype=np.float32), depth_comp=0, color_comp=2,
                     jpeg_encoder=lambda x: jpeg_bytes(x, 70, sub))
    s = SensFile(p)
    assert rg.digest(s.color(0)) == rg.expect(f"jpeg_sampling_{sub:06x}_{W}x{H}", "libref_sens.so", file_digest(p), lambda: ref_colour(p, W, H))


@pytest.mark.parametrize("mode", ["rgb", "rgba", "gray", "palette", "rgb16"])
def test_png_colour_frames_match_stb(tmp_path, built, mode):
    """TYPE_PNG colour (sensorData.h:346-351): same RGB bytes as stbi_load_from_memory(..., 3)"""
    import cv2
    rng = np.random.default_rng(5); W, H = 53, 37
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    if mode == "rgb":
        ok, buf = cv2.imencode(".png", img[:, :, ::-1])
    elif mode == "rgba":
        ok, buf = cv2.imencode(".png", np.dstack([img[:, :, ::-1], rng.integers(0, 256, (H, W), dtype=np.uint8)]))
    elif mode == "gray":
        ok, buf = cv2.imencode(".png", img[:, :, 0])
    elif mode == "rgb16":
        ok, buf = cv2.imencode(".png", (img[:, :, ::-1].astype(np.uint16) << 8) | 0x5A)
    else:
        from PIL import Image
        import io
        b = io.BytesIO(); Image.fromarray(img).quantize(37).save(b, format="PNG"); buf = np.frombuffer(b.getvalue(), np.uint8); ok = True
    assert ok
    D = np.full((1, 8, 8), 1000, np.uint16); P = np.eye(4, dtype=np.float32)[None]
    p = str(tmp_path / "p.sens")
    synth.write_sens(p, D, np.zeros((1, H, W, 3), np.uint8), P, np.eye(4, dtype=np.float32), depth_comp=0, color_comp=1,
                     jpeg_encoder=lambda x: bytes(buf))
    s = SensFile(p)
    if mode == "rgb16":                                  # stb_image v2.08 rejects 16-bit PNGs; so do we
        from scannet_b200 import ScnError
        with pytest.raises(ScnError):
            s.color(0)
        ours = rg.digest("rejected")
    else:
        ours = rg.digest(s.color(0))

    def ref():
        L = ref_lib(); r = L.ref_sens_open(p.encode())
        rc = np.zeros((H, W, 3), np.uint8); st = L.ref_sens_color(r, 0, rc.ctypes.data)
        L.ref_sens_close(r)
        return rg.digest("rejected") if st != 0 else rg.digest(rc)

    assert ours == rg.expect(f"png_{mode}", "libref_sens.so", file_digest(p), ref)


def test_writer_round_trip_through_reference(tmp_path, built):
    """scn_sens_create/add_frame/save -> the reference loads it and decodes identical depth (our deflate, its inflate)."""
    D, Cc, P, K = synth.make_frames(3, seed=4, width=96, height=64, loop_frames=30, noise_mm=1.0)
    w = SensFile.create((96, 64), (96, 64), K, K, color_compression=0, depth_compression=1)
    for f in range(3):
        w.add_frame(Cc[f], D[f], P[f], f * 33333, f * 33333)
    p = str(tmp_path / "ours.sens"); w.save(p)

    def ref():
        L = ref_lib(); r = L.ref_sens_open(p.encode()); assert r
        out = []
        for f in range(3):
            rd = np.zeros((64, 96), np.uint16); assert L.ref_sens_depth(r, f, rd.ctypes.data) == 0
            rc = np.zeros((64, 96, 3), np.uint8); assert L.ref_sens_color(r, f, rc.ctypes.data) == 0
            out += [rd, rc]
        L.ref_sens_close(r)
        return rg.digest(*out)

    # the file this writer produces is the one the reference was seen to load, and it decoded the frames that went in
    assert rg.expect("writer_round_trip", "libref_sens.so", file_digest(p), ref) == rg.digest(*[x for f in range(3) for x in (D[f], Cc[f])])
    s = SensFile(p)
    assert s.n_frames == 3 and (s.depth(1) == D[1]).all() and (s.color(2) == Cc[2]).all()
    # compression actually compresses
    assert s.frame_meta(0)[4] < 96 * 64 * 2 * 0.8
    # pose write-back + byte-identical re-save
    T = np.eye(4, dtype=np.float32); T[0, 3] = 1.5
    s.set_pose(1, T); p2 = str(tmp_path / "ours2.sens"); s.save(p2)
    s2 = SensFile(p2); assert (s2.pose(1) == T).all() and (s2.depth(2) == D[2]).all()


def cli_digest(tool, p, out):
    """stdout (paths replaced) and every file `tool <p> <out>` writes"""
    o = subprocess.run([tool, p, str(out)], capture_output=True, text=True)
    assert o.returncode == 0, o.stderr
    names = sorted(os.listdir(out))
    assert len(names) == 1 + 3 * 5
    return rg.digest(o.stdout.replace(str(out), "OUT").replace(p, "IN"), *[x for n in names for x in (n, (out / n).read_bytes())])


def test_cli_outputs_match_reference_binary(stream, tmp_path):
    """`sens <file> <outDir>`: identical _info.txt, .pose.txt, .depth.pgm, .color.jpg files and header text."""
    p = stream[0]
    ours = cli_digest(os.path.join(ROOT, "scannet_b200", "bin", "sens"), p, tmp_path / "ours")
    assert ours == rg.expect("sens_cli", "sens_ref", file_digest(p), lambda: cli_digest(REF_BIN, p, tmp_path / "ref"))


def test_errors_are_statuses_not_crashes(tmp_path, built):
    from scannet_b200 import ScnError
    with pytest.raises(ScnError):
        SensFile(str(tmp_path / "missing.sens"))
    bad = tmp_path / "bad.sens"; bad.write_bytes(b"\x03\x00\x00\x00" + b"\x00" * 64)
    with pytest.raises(ScnError) as e:
        SensFile(str(bad))
    assert "Invalid file version" in str(e.value)
    trunc = tmp_path / "trunc.sens"
    D, Cc, P, K = synth.make_frames(1, seed=1, width=32, height=24)
    synth.write_sens(str(trunc), D, Cc, P, K, depth_comp=1, color_comp=0)
    data = trunc.read_bytes(); trunc.write_bytes(data[: len(data) // 2])
    with pytest.raises(ScnError):
        SensFile(str(trunc))


@pytest.mark.parametrize("wh,n,noise,drop", [((96, 64), 4, 1.0, 0.03), ((640, 480), 2, 2.0, 0.02), ((160, 120), 3, 0.0, 0.0), ((33, 17), 2, 5.0, 0.3)])
def test_written_file_is_byte_identical_to_the_reference_writer(tmp_path, built, wh, n, noise, drop):
    """scn_sens_create/add_frame/save vs SensorData::initDefault/addFrame/saveToFile (sensorData.h:888-929,1058-1109): the
    same bytes, including the depth streams (stb_image_write's zlib writer restated decision for decision)."""
    D, Cc, P, K = synth.make_frames(n, seed=7, width=wh[0], height=wh[1], loop_frames=40, noise_mm=noise, drop=drop)
    w = SensFile.create(wh, wh, K, K, color_compression=0, depth_compression=1, sensor_name="ref_shim")
    for f in range(n):
        w.add_frame(Cc[f], D[f], P[f], f * 33333, f * 33333)
    ours = str(tmp_path / "ours.sens"); w.save(ours)
    K32 = np.ascontiguousarray(K, np.float32); Cc = np.ascontiguousarray(Cc); D = np.ascontiguousarray(D); P32 = np.ascontiguousarray(P, np.float32)

    def ref():
        L = ref_lib()
        L.ref_sens_write.argtypes = [C.c_char_p] + [C.c_uint32] * 4 + [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        r = str(tmp_path / "ref.sens")
        assert L.ref_sens_write(r.encode(), wh[0], wh[1], wh[0], wh[1], K32.ctypes.data, K32.ctypes.data, 1000.0, 1, n, Cc.ctypes.data, D.ctypes.data, P32.ctypes.data) == 0
        return file_digest(r)

    assert file_digest(ours) == rg.expect(f"sens_writer_{wh[0]}x{wh[1]}_n{n}", "libref_sens.so", rg.digest(K32, Cc, D, P32), ref)


def test_raw_colour_is_saved_as_png(tmp_path, built):
    """saveToImages on TYPE_RAW colour writes frame-XXXXXX.color.png (the name sensorData.h:1410-1440 uses) holding the same pixels."""
    import cv2
    D, Cc, P, K = synth.make_frames(2, seed=1, width=64, height=48, loop_frames=20)
    rng = np.random.default_rng(3)
    Cc = np.clip(Cc.astype(np.int32) + rng.integers(-30, 30, Cc.shape), 0, 255).astype(np.uint8)
    p = str(tmp_path / "raw.sens"); synth.write_sens(p, D, Cc, P, K, depth_comp=1, color_comp=0)
    s = SensFile(p); out = tmp_path / "img"; s.save_to_images(str(out))
    for i in range(2):
        f = out / f"frame-{i:06d}.color.png"
        assert f.exists()
        assert (cv2.imread(str(f))[:, :, ::-1] == Cc[i]).all()
    # and it is a stream this library's own PNG reader accepts: wrap it as a TYPE_PNG .sens
    q = str(tmp_path / "png.sens")
    png = [(out / f"frame-{i:06d}.color.png").read_bytes() for i in range(2)]
    synth.write_sens(q, D, Cc, P, K, depth_comp=1, color_comp=1, jpeg_encoder=lambda rgb, _it=iter(png): next(_it))
    t = SensFile(q)
    assert (t.color(0) == Cc[0]).all() and (t.color(1) == Cc[1]).all()


def _decode_matches_reference(tmp_path, key, payload, W, H, comp):
    """this library's decode of one colour payload == the reference's (which must decode it too)"""
    D = np.full((1, 8, 8), 1000, np.uint16); P = np.eye(4, dtype=np.float32)[None]
    p = str(tmp_path / "x.sens")
    synth.write_sens(p, D, np.zeros((1, H, W, 3), np.uint8), P, np.eye(4, dtype=np.float32), depth_comp=0, color_comp=comp, jpeg_encoder=lambda x: payload)
    return rg.digest(SensFile(p).color(0)) == rg.expect(key, "libref_sens.so", file_digest(p), lambda: ref_colour(p, W, H))


@pytest.mark.parametrize("wh,q,sub,rst,gray", [((64, 48), 85, None, 0, False), ((160, 120), 90, 0x221111, 0, False), ((161, 119), 75, 0x111111, 0, False),
                                              ((97, 33), 50, 0x211111, 0, False), ((200, 150), 95, 0x221111, 7, False), ((33, 17), 30, 0x121111, 0, False),
                                              ((75, 41), 60, None, 3, True)])
def test_progressive_jpeg_matches_stb(tmp_path, built, wh, q, sub, rst, gray):
    """SOF2: spectral selection + successive approximation (stb_image.h:1771-1913, 2582-2600), DC/AC first and refinement passes,
    interleaved DC scans, non-interleaved AC scans, restart intervals."""
    import cv2
    W, H = wh; rng = np.random.default_rng(W * H + q)
    yy, xx = np.mgrid[0:H, 0:W]
    img = np.stack([(xx * 255 // max(W - 1, 1)), (yy * 255 // max(H - 1, 1)), ((xx + yy) % 256)], -1).astype(np.int32) + rng.integers(-25, 25, (H, W, 3))
    img = np.clip(img, 0, 255).astype(np.uint8)
    params = [int(cv2.IMWRITE_JPEG_QUALITY), q, int(cv2.IMWRITE_JPEG_PROGRESSIVE), 1]
    if sub is not None: params += [int(cv2.IMWRITE_JPEG_SAMPLING_FACTOR), sub]
    if rst: params += [int(cv2.IMWRITE_JPEG_RST_INTERVAL), rst]
    ok, buf = cv2.imencode(".jpg", img[:, :, 0] if gray else img[:, :, ::-1], params)
    assert ok and b"\xff\xc2" in buf.tobytes()
    assert _decode_matches_reference(tmp_path, f"progressive_{W}x{H}_q{q}_{sub}_rst{rst}_{'gray' if gray else 'rgb'}", buf.tobytes(), W, H, 2)


def _png(img, interlace, depth=8, ctype=2, palette=None, filt=0):
    """minimal PNG writer for the test (Adam7 when interlace): rows use filter `filt` in {0, 1, 2}"""
    import struct, zlib
    H, W = img.shape[:2]
    def chunk(t, d): return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xFFFFFFFF)
    def pack_rows(sub):
        h, w = sub.shape[:2]
        if depth == 8: rows = sub.reshape(h, -1).astype(np.uint8)
        else:
            bits = np.unpackbits(sub.reshape(h, w, 1).astype(np.uint8), axis=2)[:, :, 8 - depth:].reshape(h, -1)
            rows = np.packbits(bits, axis=1)
        bpp = max(1, rows.shape[1] // max(w, 1)) if depth == 8 else 1
        out = b""; prev = np.zeros(rows.shape[1], np.uint8)
        for r in rows:
            if filt == 1: left = np.concatenate([np.zeros(bpp, np.uint8), r[:-bpp]]); enc = (r.astype(int) - left) % 256
            elif filt == 2: enc = (r.astype(int) - prev) % 256
            else: enc = r
            out += bytes([filt]) + enc.astype(np.uint8).tobytes(); prev = r
        return out
    if interlace:
        raw = b""
        for x0, y0, dx, dy in [(0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)]:
            sub = img[y0::dy, x0::dx]
            if sub.shape[0] and sub.shape[1]: raw += pack_rows(sub)
    else: raw = pack_rows(img)
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, depth, ctype, 0, 0, 1 if interlace else 0))
    if palette is not None: out += chunk(b"PLTE", palette.astype(np.uint8).tobytes())
    return out + chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b"")


@pytest.mark.parametrize("wh", [(53, 37), (8, 8), (3, 2), (1, 1), (17, 5)])
@pytest.mark.parametrize("kind", ["rgb", "rgba", "gray", "gray4", "pal2"])
def test_interlaced_png_matches_stb(tmp_path, built, wh, kind):
    """Adam7 (stb_image.h:4310-4350), incl. images smaller than the 8x8 lattice and sub-byte depths"""
    W, H = wh; rng = np.random.default_rng(W * 100 + H)
    pal = None
    if kind == "rgb": img, depth, ct = rng.integers(0, 256, (H, W, 3)), 8, 2
    elif kind == "rgba": img, depth, ct = rng.integers(0, 256, (H, W, 4)), 8, 6
    elif kind == "gray": img, depth, ct = rng.integers(0, 256, (H, W)), 8, 0
    elif kind == "gray4": img, depth, ct = rng.integers(0, 16, (H, W)), 4, 0
    else: img, depth, ct, pal = rng.integers(0, 4, (H, W)), 2, 3, rng.integers(0, 256, (4, 3))
    # stb_image v2.08 computes `prior` before it moves `cur` to the packed bytes of a sub-byte-depth row (stb_image.h:4003-4012),
    # so its up/avg/paeth filters read uninitialised memory there: only none/sub are defined in the reference at depth < 8
    # (this library follows the PNG specification for the others)
    for filt in ((0, 1, 2) if depth == 8 else (0, 1)):
        assert _decode_matches_reference(tmp_path, f"png_adam7_{kind}_{W}x{H}_filter{filt}", _png(img.astype(np.uint8), True, depth, ct, pal, filt), W, H, 1), (kind, filt)
    assert _decode_matches_reference(tmp_path, f"png_plain_{kind}_{W}x{H}_filter1", _png(img.astype(np.uint8), False, depth, ct, pal, 1), W, H, 1)   # and the plain layout through the same writer


@pytest.mark.parametrize("cache,threads", [(1, 1), (3, 2), (16, 0), (64, 8)])
def test_read_ahead_cache_returns_the_stream_in_order(stream, cache, threads):
    """RGBDFrameCacheRead counterpart: same frames as the random-access decode, in order, for any cache size / thread count"""
    p, D, Cc, P, K = stream
    s = SensFile(p)
    got = list(s.read_ahead(cache, threads))
    assert len(got) == s.n_frames
    for i, (d, c, td, tc) in enumerate(got):
        assert (d == s.depth(i)).all() and (c == s.color(i)).all()
        assert (td, tc) == (s.frame_meta(i)[2], s.frame_meta(i)[1])


def test_read_ahead_cache_early_exit_and_errors(stream, tmp_path):
    from scannet_b200 import ScnError
    p = stream[0]
    s = SensFile(p)
    it = s.read_ahead(2, 2); next(it); it.close()                      # destroyed while workers are mid-stream
    raw = bytearray(open(p, "rb").read())
    # corrupt the zlib header of the LAST frame's depth payload (the file ends: ..., color payload, depth payload, u64 numIMU = 0)
    n_depth = s.frame_meta(s.n_frames - 1)[4]
    raw[len(raw) - 8 - n_depth] ^= 0xFF
    q = tmp_path / "bad.sens"; q.write_bytes(bytes(raw))
    t = SensFile(str(q)); it = t.read_ahead(4, 2)
    for _ in range(t.n_frames - 1):
        next(it)
    with pytest.raises(ScnError, match="corrupt zlib depth stream"):
        next(it)


def test_simd_and_scalar_idct_give_the_same_bytes(tmp_path, built):
    """the AVX2 IDCT against the scalar one (SCN_JPEG_SCALAR=1) on clean, extreme and corrupted JPEG payloads, in two child
    processes (the switch is read once per process): same status and same pixels for every payload"""
    import cv2, pickle, sys
    rng = np.random.default_rng(9); W, H = 96, 72
    payloads = []
    for q in (100, 75, 20, 3):
        for kind in ("noise", "smooth", "binary"):
            if kind == "noise": img = rng.integers(0, 256, (H, W, 3))
            elif kind == "smooth": xx, yy = np.meshgrid(np.arange(W), np.arange(H)); img = np.stack([xx, yy, np.zeros((H, W))], -1) * 2
            else: img = (rng.integers(0, 2, (H, W, 3)) * 255)
            for prog in (0, 1):
                payloads.append(cv2.imencode(".jpg", img.astype(np.uint8), [int(cv2.IMWRITE_JPEG_QUALITY), q, int(cv2.IMWRITE_JPEG_PROGRESSIVE), prog])[1].tobytes())
    clean = list(payloads)
    for p in clean:                                              # corrupt the entropy-coded part: wild coefficients, early markers
        for _ in range(6):
            b = bytearray(p)
            for _ in range(int(rng.integers(1, 6))):
                b[int(rng.integers(len(b) // 2, len(b) - 2))] = int(rng.integers(0, 255))
            payloads.append(bytes(b))
    D = np.full((len(payloads), 8, 8), 1000, np.uint16); P = np.tile(np.eye(4, dtype=np.float32), (len(payloads), 1, 1))
    f = str(tmp_path / "many.sens"); it = iter(payloads)
    synth.write_sens(f, D, np.zeros((len(payloads), H, W, 3), np.uint8), P, np.eye(4, dtype=np.float32), depth_comp=0, color_comp=2, jpeg_encoder=lambda x: next(it))
    code = ("import sys, pickle, numpy as np; sys.path.insert(0, %r)\n"
            "from scannet_b200.sens import SensFile\nfrom scannet_b200 import ScnError\n"
            "s = SensFile(%r); out = []\n"
            "for i in range(s.n_frames):\n"
            "    try: out.append(s.color(i).tobytes())\n"
            "    except ScnError as e: out.append(str(e))\n"
            "pickle.dump(out, open(sys.argv[1], 'wb'))\n") % (ROOT, f)
    res = {}
    for mode in ("simd", "scalar"):
        o = str(tmp_path / (mode + ".pkl"))
        env = dict(os.environ); env.pop("SCN_JPEG_SCALAR", None)
        if mode == "scalar": env["SCN_JPEG_SCALAR"] = "1"
        r = subprocess.run([sys.executable, "-c", code, o], env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-1500:]
        res[mode] = pickle.load(open(o, "rb"))
    assert len(res["simd"]) == len(payloads)
    assert sum(isinstance(x, bytes) for x in res["simd"]) >= len(clean)
    assert res["simd"] == res["scalar"]


def test_oversubscribed_jpeg_huffman_table_is_rejected_before_any_table_write(tmp_path, built):
    """ADVICE r01 (high): a DHT segment with counts[0]=200 used to index far outside the 512-entry fast table.  The decoder must
    refuse it like stb_image does (bad code lengths), and a SOF whose size disagrees with the container must fail before any
    plane is sized from the in-stream values."""
    import cv2
    from scannet_b200 import ScnError
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (16, 16, 3), dtype=np.uint8)
    ok, buf = cv2.imencode(".jpg", img, [int(cv2.IMWRITE_JPEG_QUALITY), 80]); assert ok
    good = bytes(buf)
    i = good.index(b"\xff\xc4")                                           # first DHT segment
    bad = bytearray(good); bad[i + 5] = 200                               # counts[0] = 200 codes of length 1
    j = good.index(b"\xff\xc0")                                           # SOF0: claim a 65535 x 65535 image
    huge = bytearray(good); huge[j + 5:j + 9] = b"\xff\xff\xff\xff"
    D = np.full((1, 8, 8), 1000, np.uint16); P = np.eye(4, dtype=np.float32)[None]
    for name, payload in (("dht", bad), ("sof", huge)):
        p = str(tmp_path / f"{name}.sens")
        synth.write_sens(p, D, np.zeros((1, 16, 16, 3), np.uint8), P, np.eye(4, dtype=np.float32), depth_comp=0, color_comp=2,
                         jpeg_encoder=lambda x, _b=bytes(payload): _b)
        s = SensFile(p)
        with pytest.raises(ScnError):
            s.color(0)


def test_pose_write_back_over_the_opened_file_and_unmapped_open(tmp_path, built, monkeypatch):
    """An opened stream points into the mapped file: saving over that very file (the pose write-back workflow) must not
    truncate the mapping, and the read-whole fallback (SCN_SENS_NO_MMAP) gives the same bytes."""
    D, Cc, P, K = synth.make_frames(4, seed=9, width=96, height=64, loop_frames=30, noise_mm=1.0)
    w = SensFile.create((96, 64), (96, 64), K, K, color_compression=0, depth_compression=1)
    for f in range(4):
        w.add_frame(Cc[f], D[f], P[f], f, f)
    p = str(tmp_path / "scan.sens"); w.save(p)
    before = open(p, "rb").read()
    s = SensFile(p)
    T = np.eye(4, dtype=np.float32); T[1, 3] = -2.25
    s.set_pose(2, T)
    s.save(p)                                             # over the input
    assert (s.depth(3) == D[3]).all() and (s.color(0) == Cc[0]).all()      # the old mapping is still intact
    after = open(p, "rb").read()
    assert len(after) == len(before) and after != before
    assert not [f for f in os.listdir(tmp_path) if ".tmp" in f]
    s2 = SensFile(p)
    assert (s2.pose(2) == T).all() and (s2.pose(1) == P[1]).all() and (s2.depth(0) == D[0]).all()
    monkeypatch.setenv("SCN_SENS_NO_MMAP", "1")
    s3 = SensFile(p)
    assert s3.n_frames == 4 and (s3.pose(2) == T).all()
    for f in range(4):
        assert (s3.depth(f) == D[f]).all() and (s3.color(f) == Cc[f]).all()
    p3 = str(tmp_path / "copy.sens"); s3.save(p3)
    assert open(p3, "rb").read() == after
