"""GPU parity for R4 (colour decode): JPEG frames decoded on the device (scannet_b200/csrc/jpeg_gpu.cu) must be byte-identical
to the host decoder (jpeg.cpp), which tests/test_sens_cpu.py pins byte for byte against the reference's stb_image
(sensorData.h:609-616 -> stb_image.h) — and to the reference's own decode of the same streams (stored digests,
reference_golden.py).
Matrix: the sampling modes the device path takes itself (4:4:4, 4:2:2, 4:2:0, 4:4:0, grey), restart intervals, odd sizes, the
ScanNet colour size 1296x968, a depth-registered sampling map; progressive / corrupt frames must come back through the host
decoder with the same bytes / the same error."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import reference_golden as rg
from scannet_b200 import ScnError, sens, synth
from scannet_b200.sens import SensFile

pytestmark = pytest.mark.gpu
REF_SO = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libref_sens.so")


def image(W, H, seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    img = np.stack([(xx * 255 // max(W - 1, 1)), (yy * 255 // max(H - 1, 1)), ((xx * 3 + yy * 5) % 256)], -1).astype(np.int32)
    img += rng.integers(-30, 30, (H, W, 3))
    img[H // 3: H // 2, W // 4: W // 2] = rng.integers(0, 256, 3)              # a flat patch: long zero runs / EOB-only blocks
    return np.clip(img, 0, 255).astype(np.uint8)


def encode(img, q=85, sub=None, rst=0, gray=False, progressive=False):
    import cv2
    params = [int(cv2.IMWRITE_JPEG_QUALITY), q]
    if sub is not None: params += [int(cv2.IMWRITE_JPEG_SAMPLING_FACTOR), sub]
    if rst: params += [int(cv2.IMWRITE_JPEG_RST_INTERVAL), rst]
    if progressive: params += [int(cv2.IMWRITE_JPEG_PROGRESSIVE), 1]
    ok, buf = cv2.imencode(".jpg", img[:, :, 0] if gray else img[:, :, ::-1], params)
    assert ok
    return buf.tobytes()


def host_decode(tmp_path, jpegs, W, H, name="h.sens", ref_key=None):
    """the product's host decoder through a .sens container; checked against the reference's decode when ref_key is given"""
    D = np.full((len(jpegs), 8, 8), 1000, np.uint16); P = np.tile(np.eye(4, dtype=np.float32), (len(jpegs), 1, 1))
    p = str(tmp_path / name)
    it = iter(jpegs)
    synth.write_sens(p, D, np.zeros((len(jpegs), H, W, 3), np.uint8), P, np.eye(4, dtype=np.float32), depth_comp=0, color_comp=2,
                     jpeg_encoder=lambda x: next(it))
    s = SensFile(p)
    out = np.stack([s.color(i) for i in range(len(jpegs))])
    if ref_key is not None:
        def ref():
            L = C.CDLL(REF_SO); L.ref_sens_open.restype = C.c_void_p; L.ref_sens_open.argtypes = [C.c_char_p]
            L.ref_sens_color.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]; L.ref_sens_close.argtypes = [C.c_void_p]
            r = L.ref_sens_open(p.encode()); frames = []
            for i in range(len(jpegs)):
                rc = np.zeros((H, W, 3), np.uint8)
                assert L.ref_sens_color(r, i, rc.ctypes.data) == 0
                frames.append(rc)
            L.ref_sens_close(r)
            return rg.digest(np.stack(frames))
        with open(p, "rb") as fh:
            inputs = rg.digest(fh.read())
        assert rg.digest(out) == rg.expect(ref_key, "libref_sens.so", inputs, ref), "host decoder differs from the reference (stb_image)"
    return s, out


CASES = [((64, 48), 85, None, 0, False), ((160, 120), 90, 0x221111, 0, False), ((161, 119), 75, 0x111111, 0, False),
         ((97, 33), 50, 0x211111, 0, False), ((200, 150), 95, 0x221111, 7, False), ((33, 17), 30, 0x121111, 0, False),
         ((75, 41), 60, None, 3, True), ((17, 9), 99, 0x221111, 1, False), ((640, 480), 80, 0x221111, 0, False), ((8, 8), 10, 0x221111, 0, False)]


@pytest.mark.parametrize("wh,q,sub,rst,gray", CASES)
def test_device_jpeg_is_byte_identical(tmp_path, built, wh, q, sub, rst, gray):
    W, H = wh
    jpegs = [encode(image(W, H, 10 * i + W), q, sub, rst, gray) for i in range(3)]
    s, ref = host_decode(tmp_path, jpegs, W, H, ref_key=f"device_jpeg_{W}x{H}_q{q}_{sub}_rst{rst}_{'gray' if gray else 'rgb'}")
    out = torch.zeros((3, H, W, 3), dtype=torch.uint8, device="cuda")
    k = sens.jpeg_decode_batch_device(jpegs, W, H, out.data_ptr())
    assert k == 3, "these streams are baseline single-scan JPEG: the device must decode them itself"
    assert (out.cpu().numpy() == ref).all()
    out2 = torch.zeros((3, H, W, 3), dtype=torch.uint8, device="cuda")      # the .sens entry point
    assert s.decode_color_device(0, 3, out2.data_ptr()) == 3
    assert (out2.cpu().numpy() == ref).all()


def test_scannet_colour_size_and_registered_sampling(tmp_path, built):
    """1296x968 colour (ScannerApp/README.md:20-23) + the depth-pixel -> colour-pixel map of the fusion path"""
    W, H = 1296, 968
    jpegs = [encode(image(W, H, i), 80, 0x221111) for i in range(4)]
    s, ref = host_decode(tmp_path, jpegs, W, H, ref_key="device_jpeg_scannet_colour")
    out = torch.zeros((4, H, W, 3), dtype=torch.uint8, device="cuda")
    assert sens.jpeg_decode_batch_device(jpegs, W, H, out.data_ptr()) == 4
    assert (out.cpu().numpy() == ref).all()
    rng = np.random.default_rng(1)
    lut = rng.integers(-1, W * H, 640 * 480).astype(np.int32); lut[:7] = [-1, 0, W - 1, W, W * H - 1, W * (H - 1), 2 * W - 1]
    d_lut = torch.from_numpy(lut).cuda()
    reg = torch.zeros((4, 640 * 480, 3), dtype=torch.uint8, device="cuda")
    assert sens.jpeg_decode_batch_device(jpegs, W, H, reg.data_ptr(), d_lut.data_ptr(), 640 * 480) == 4
    want = ref.reshape(4, W * H, 3)[:, np.maximum(lut, 0)]; want[:, lut < 0] = 0
    assert (reg.cpu().numpy() == want).all()


def test_streams_the_device_declines_go_through_the_host_decoder(tmp_path, built):
    """a progressive frame and a non-interleaved-friendly odd sampling in the middle of a batch: same bytes, device count says so"""
    W, H = 120, 88
    jpegs = [encode(image(W, H, 1), 85, 0x221111), encode(image(W, H, 2), 85, 0x221111, progressive=True), encode(image(W, H, 3), 70, 0x411111),
             encode(image(W, H, 4), 60, 0x111111, rst=2)]
    s, ref = host_decode(tmp_path, jpegs, W, H, ref_key="device_jpeg_declined_streams")
    out = torch.zeros((4, H, W, 3), dtype=torch.uint8, device="cuda")
    k = sens.jpeg_decode_batch_device(jpegs, W, H, out.data_ptr())
    assert k == 2
    assert (out.cpu().numpy() == ref).all()


def test_corrupt_frames_behave_like_the_host_decoder(tmp_path, built):
    W, H = 96, 64
    good = encode(image(W, H, 5), 85, 0x221111)
    cut = good[: len(good) * 2 // 3]                                          # truncated scan: the host decoder still returns an image (stb reports "no EOI")
    wrong_size = encode(image(W + 8, H, 6), 85, 0x221111)                     # header says another size: an error on both paths
    s, ref = host_decode(tmp_path, [good, cut], W, H)                         # device path == host path of this library on damaged input
    out = torch.zeros((2, H, W, 3), dtype=torch.uint8, device="cuda")
    sens.jpeg_decode_batch_device([good, cut], W, H, out.data_ptr())
    assert (out.cpu().numpy() == ref).all()
    with pytest.raises(ScnError):
        sens.jpeg_decode_batch_device([good, wrong_size], W, H, out.data_ptr())


def test_many_frames_in_one_launch(tmp_path, built):
    """more frames than resident warps per SM x SMs would hold at once is not needed for correctness, but mixed table sets are:
    two qualities (two DQT sets) interleaved in one batch"""
    W, H = 160, 120
    jpegs = [encode(image(W, H, i), 60 + 30 * (i & 1), 0x221111 if i % 3 else 0x211111) for i in range(96)]
    s, ref = host_decode(tmp_path, jpegs, W, H, ref_key="device_jpeg_mixed_tables_96")
    out = torch.zeros((96, H, W, 3), dtype=torch.uint8, device="cuda")
    assert sens.jpeg_decode_batch_device(jpegs, W, H, out.data_ptr()) == 96
    assert (out.cpu().numpy() == ref).all()
