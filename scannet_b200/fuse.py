"""Host-side mirror of the scene fusion driver (``scn_fuse_scene`` / ``scn_fuse_many``): the contract of the reference's external
reconstruction stage (/root/reference/Server/scan_processor.py:27-35,123-138) — a ``.sens`` file in, a fused volume and
``<id>_vh.ply`` out — one scene per GPU (/root/reference/Server/process.py:75).  All work happens in libscannet_b200.so."""
from __future__ import annotations

import ctypes as C

from ._lib import check, lib
from .tsdf import default_params


class FuseReport(C.Structure):
    _fields_ = [("status", C.c_int32), ("device", C.c_int32), ("gpu_decode", C.c_int32), ("volume_reused", C.c_uint32), ("color_frames_on_device", C.c_uint32),
                ("frames_integrated", C.c_uint64), ("frames_skipped", C.c_uint64), ("frames_skipped_pose", C.c_uint64),
                ("blocks_allocated", C.c_uint64), ("voxels_updated", C.c_uint64),
                ("mesh_vertices", C.c_uint64), ("mesh_faces", C.c_uint64), ("device_bytes_in_use", C.c_uint64),
                ("fuse_s", C.c_double), ("decode_wait_s", C.c_double), ("depth_decode_s", C.c_double), ("color_decode_s", C.c_double),
                ("integrate_s", C.c_double), ("depth_pack_s", C.c_double), ("depth_kernel_s", C.c_double),
                ("color_host_s", C.c_double), ("color_entropy_s", C.c_double), ("color_convert_s", C.c_double), ("setup_s", C.c_double), ("buffers_s", C.c_double), ("teardown_s", C.c_double),
                ("mc_s", C.c_double), ("ply_s", C.c_double), ("total_s", C.c_double)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["frames_per_s_incl_decode"] = d["frames_integrated"] / d["fuse_s"] if d["fuse_s"] > 0 else 0.0
        return d


def fuse_scene(sens_path: str, out_ply: str | None = None, device: int = 0, decode_mode: str | None = None, **param_over) -> dict:
    params = default_params(**param_over)
    rep = FuseReport()
    check(lib().scn_fuse_scene(str(sens_path).encode(), str(out_ply).encode() if out_ply else None, C.byref(params), C.c_int(device),
                               decode_mode.encode() if decode_mode else None, C.byref(rep)))
    return rep.as_dict()


def fuse_many(sens_paths, out_plys=None, devices=(0,), decode_mode: str | None = None, **param_over):
    params = default_params(**param_over)
    n = len(sens_paths)
    sp = (C.c_char_p * n)(*[str(p).encode() for p in sens_paths])
    op = (C.c_char_p * n)(*[(str(p).encode() if p else None) for p in (out_plys or [None] * n)])
    dv = (C.c_int * len(devices))(*devices)
    reps = (FuseReport * n)()
    check(lib().scn_fuse_many(sp, op, C.c_uint32(n), C.byref(params), dv, C.c_uint32(len(devices)),
                              decode_mode.encode() if decode_mode else None, reps))
    return [r.as_dict() for r in reps]
