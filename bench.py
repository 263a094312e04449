#!/usr/bin/env python
"""bench.py — headline benchmark of the ScanNet hot path on B200.

Metric (BASELINE.json): depth frames/s integrated (640x480, 4 mm voxel) into the hashed TSDF,
plus the HBM roofline fraction of the dominant kernel.  Workload = BASELINE.json configs[1]
("synthetic 640x480 .sens, 1000 frames, 4 mm TSDF"): a seeded box-room RGB-D stream
(scannet_b200/synth.py conventions) rendered on the device with torch (data generation only).

A "step" = fusing the next --frames-per-step frames of the stream into the volume through the
C ABI (include/scannet_b200.h).  Two timed passes over the same K steps:
  value : frames already resident in HBM  -> scn_tsdf_integrate_device
  e2e   : frames in pinned HOST memory    -> scn_tsdf_integrate_batch (H2D inside the timed region)
          + a device->host read of the step's result (scn_tsdf_stats counters).
N>1 (torchrun): one scene per rank/GPU, no data-path collective (SURVEY.md §8e); NCCL is only the
barrier + max-over-ranks reduction of the device-measured time.  `--impl reference` times the CPU
statement of the same path (oracle/tsdf_oracle.c — the reference ships no TSDF code) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

# stdout carries exactly ONE line (the JSON result): everything else that C libraries print on fd 1 (NCCL's version banner,
# the reference's printf) is diverted to stderr for the life of the process.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


METRIC = "depth frames/sec integrated (640x480, 4 mm voxel)"
UNIT = "frames/s"
W, H = 640, 480


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------- synthetic stream
def scene_poses(n, seed, loop):
    from scannet_b200 import synth
    # every rank fuses its own scene (different sphere layout per seed) in a room of the same size along the same
    # camera loop, so per-GPU work is the same to within a few percent and the N-GPU numbers measure scaling, not scenes
    sc = synth.BoxRoomScene(size=(6.0, 5.0, 3.0), seed=seed, width=W, height=H)
    P = np.stack([sc.camera_pose(i, loop) for i in range(n)]).astype(np.float32)
    return sc, P


def render_depth_torch(sc, P, device, chunk=50):
    """Same analytic scene as synth.BoxRoomScene.render, evaluated with torch on `device`.
    Returns uint16 depth [N,H,W] (mm).  Data generation only — not part of any timed region."""
    import torch
    N = len(P)
    out = torch.empty((N, sc.H, sc.W), dtype=torch.int16, device=device)
    rays = torch.as_tensor(sc.rays_cam, dtype=torch.float64, device=device)          # [H,W,3]
    size = torch.as_tensor(sc.size, dtype=torch.float64, device=device)
    for s in range(0, N, chunk):
        T = torch.as_tensor(P[s:s + chunk], dtype=torch.float64, device=device)
        R, o = T[:, :3, :3], T[:, :3, 3]
        d = torch.einsum("hwj,nij->nhwi", rays, R)                                     # [n,H,W,3]
        tb = torch.full(d.shape[:3], float("inf"), dtype=torch.float64, device=device)
        for ax in range(3):
            for wall in (0.0, float(size[ax])):
                t = (wall - o[:, None, None, ax]) / d[..., ax]
                hit = (t > 1e-6) & (t < tb)
                tb = torch.where(hit, t, tb)
        for c, r in sc.spheres:
            cc = torch.as_tensor(c, dtype=torch.float64, device=device)
            oc = o - cc
            a = (d * d).sum(-1); b = 2.0 * torch.einsum("nhwi,ni->nhw", d, oc); c0 = (oc * oc).sum(-1) - r * r
            disc = b * b - 4 * a * c0[:, None, None]
            t = (-b - torch.sqrt(torch.clamp(disc, min=0.0))) / (2 * a)
            hit = (disc > 0) & (t > 1e-6) & (t < tb)
            tb = torch.where(hit, t, tb)
        mm = torch.clamp(torch.round(tb * 1000.0), 0, 65535)
        mm = torch.where(torch.isfinite(tb), mm, torch.zeros_like(mm))
        out[s:s + chunk] = mm.to(torch.int32).to(torch.int16)       # bit pattern of uint16
    return out


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index; self.rows = []; self.proc = None; self.th = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None; return
        self.th = threading.Thread(target=self._read, daemon=True); self.th.start()

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = []; mx = None; reasons = set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------- shared config
SCENE_FRAMES = 1000          # BASELINE.json configs[1]: one synthetic scene = 1000 frames


def make_config(args, world):
    """The same dict in both arms (the driver compares them)."""
    SCENE_FRAMES = args.scene_frames
    n_sc = max(1, args.frames_per_step // SCENE_FRAMES)
    return {"workload": f"synthetic 640x480 .sens-style stream, {SCENE_FRAMES}-frame scenes, 4 mm hashed TSDF (BASELINE.json configs[1]); "
                        f"one step = {n_sc} fresh scene(s) fused from an empty volume (reset + {n_sc * SCENE_FRAMES} frames)",
            "frames_per_step": n_sc * SCENE_FRAMES, "scene_frames": SCENE_FRAMES, "scenes_per_step": n_sc,
            "voxel_m": 0.004, "truncation_m": "0.02+0.01*d", "batch_frames": args.batch, "scenes": world,
            "parallelism": f"one scene stream per GPU x{world}, no data-path collective",
            "l2": f"inputs larger than L2: {n_sc * SCENE_FRAMES * W * H * 2 / 1e6:.0f} MB of distinct depth per step + ~60 MB of voxel blocks per frame; no flush",
            "color": bool(args.color)}


def bench_params():
    from scannet_b200._lib import TsdfParams
    p = TsdfParams(); p.voxel_size = 0.004; p.trunc_base = 0.02; p.trunc_scale = 0.01; p.depth_min = 0.1
    p.depth_max = 6.0; p.max_integration_distance = 4.0; p.weight_sample = 1; p.weight_max = 255
    p.width = W; p.height = H; p.depth_shift = 1000.0
    return p


# ----------------------------------------------------------------------------- CPU arm
def _omp_env():
    # must be set before libgomp starts its pool: threads stay on their cores and spin between the two parallel regions of a frame
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_WAIT_POLICY", "active")


class CpuStream:
    """The CPU statement of the path (oracle/tsdf_oracle.c — the reference ships no TSDF source) fed with consecutive frames
    of rank 0's first scene, rendered on the host."""

    def __init__(self, args, threads):
        import oracle_bindings as ob
        self.ob = ob
        self.sc, _ = scene_poses(1, 0, args.loop)
        self.loop = args.loop
        self.K = self.sc.intrinsics()
        self.o = ob.OracleTsdf(bench_params(), threads=threads)
        self.pos = 0

    def run(self, n):
        """renders n frames (untimed), then times their fusion; returns seconds"""
        P = [self.sc.camera_pose(self.pos + i, self.loop).astype(np.float32) for i in range(n)]
        D = [self.sc.render(P[i])[0] for i in range(n)]
        t0 = time.perf_counter()
        for i in range(n):
            self.o.integrate(D[i], None, P[i], self.K)
        dt = time.perf_counter() - t0
        self.pos += n
        return dt

    def close(self):
        self.o.close()


def pick_threads(args):
    """'all the host threads it can use': the oracle's per-frame parallel regions stop scaling (and cross-socket traffic hurts)
    long before 128 hardware threads, so a 3-frame probe picks the best of {all, 1/2, 1/4, 1/8, 1/16} of the logical CPUs (the
    box is shared: in one run 16 threads gave 124 frames/s and 128 threads 29)."""
    n = os.cpu_count() or 1
    cands = sorted({max(1, n), max(1, n // 2), max(1, n // 4), max(1, n // 8), max(1, n // 16)}, reverse=True)
    best, best_fps, probe = cands[0], 0.0, {}
    for th in cands:
        c = CpuStream(args, th)
        c.run(1)
        fps = 3 / c.run(3)
        c.close()
        probe[str(th)] = round(fps, 2)
        if fps > best_fps:
            best, best_fps = th, fps
    return best, probe


def cpu_arm(args, steps=1, warmup=0, threads=None):
    """Bounded sample: every step fuses --cpu-frames consecutive frames of the same synthetic stream (640x480, 4 mm) into the
    growing volume; returns the cpu_baseline object + (total frames, total seconds, ms per sampled step)."""
    _omp_env()
    probe = None
    if threads is None:
        threads, probe = pick_threads(args)
    c = CpuStream(args, threads)
    c.run(1)                                                   # first frame allocates the visible blocks
    for _ in range(warmup):
        c.run(args.cpu_frames)
    dts = [c.run(args.cpu_frames) for _ in range(steps)]
    c.close()
    c1 = CpuStream(args, 1)
    c1.run(1)
    fps1 = 3 / c1.run(3)
    c1.close()
    tot = sum(dts)
    cb = {"value": steps * args.cpu_frames / tot, "unit": UNIT, "cores": threads, "kind": "port",
          "value_1thread": fps1, "host_logical_cpus": os.cpu_count(), "thread_probe_fps": probe,
          "omp": {k: os.environ.get(k) for k in ("OMP_PROC_BIND", "OMP_PLACES", "OMP_WAIT_POLICY")},
          "sample": f"{steps} step(s) x {args.cpu_frames} consecutive 640x480 frames of rank 0's first scene after {1 + warmup * args.cpu_frames} "
                    f"untimed frame(s); oracle/tsdf_oracle.c (own restatement: the reference tree has no TSDF source), OpenMP over pixels "
                    f"(allocation) and blocks (integration)"}
    return cb, 1e3 * tot / steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    cb, ms_step = cpu_arm(args, steps=args.steps, warmup=args.warmup)
    v = cb["value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args, args.gpus),
            "sampled": True, "sample_frames_per_step": args.cpu_frames,
            "cpu_baseline": cb, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    emit(line)


# ----------------------------------------------------------------------------- Segmentator side benchmark
def seg_bench(c5: bool):
    """BASELINE.json configs[0]/[4]: Segmentator on a ~50k-vertex (and optionally 2M-vertex) mesh, GPU path vs the
    reference CPU code (oracle/_ref built from the unmodified reference when present, else the C restatement)."""
    import tempfile
    import oracle_bindings as ob
    from scannet_b200 import segmentator, synth
    out = {}
    for name, (nx, ny) in ([("c1_50k", (250, 200))] + ([("c5_2m", (1600, 1250))] if c5 else [])):
        xyz, tri = synth.make_feature_mesh(nx, ny, seed=5)
        segmentator.segment_mesh(xyz[:3000], tri[(tri < 3000).all(1)])            # warm-up (context, allocator)
        runs = []
        for _ in range(3):
            t0 = time.perf_counter(); seg = segmentator.segment_mesh(xyz, tri); dt = time.perf_counter() - t0
            ms, launches = segmentator.last_timings(); runs.append((dt, ms, launches))
        runs.sort(key=lambda r: r[0]); dt, ms, launches = runs[1]
        t0 = time.perf_counter(); ref = ob.oracle_segment(xyz, tri); t_port = time.perf_counter() - t0
        rec = {"verts": int(len(xyz)), "faces": int(len(tri)), "segments": int(len(set(seg.tolist()))), "bit_identical_to_cpu": bool((seg == ref).all()),
               "gpu_path_s": dt, "stages_ms": {k: round(v, 3) for k, v in zip(["h2d", "normals", "weights", "sort", "kruskal_host", "small_merge_host", "gather_d2h_labels", "total"], ms)},
               "sort_kernel_launches": launches, "cpu_port_s": t_port, "cpu_port_kind": "oracle/seg_oracle.c -O2, 1 thread, arrays in memory"}
        # S5 on the device (SCN_SEG_DEVICE_UNIONFIND, csrc/seg.cu:k_kruskal_window) against the default host loop, same records
        try:
            segmentator.segment_mesh(xyz, tri, flags=segmentator.DEVICE_UNIONFIND)
            t0 = time.perf_counter(); seg_d = segmentator.segment_mesh(xyz, tri, flags=segmentator.DEVICE_UNIONFIND); dt_d = time.perf_counter() - t0
            ms_d, _ = segmentator.last_timings()
            rec["unionfind_device_vs_host"] = {"kruskal_device_ms": round(ms_d[4], 3), "kruskal_host_ms": round(ms[4], 3), "device_rounds": segmentator.last_uf_rounds(),
                                               "ids_identical": bool((seg_d == seg).all()), "gpu_path_s_with_device_unionfind": dt_d,
                                               "default": "host loop" }
        except Exception as e:
            rec["unionfind_device_vs_host"] = {"error": repr(e)}
        ref_bin = os.path.join(ROOT, "oracle", "_ref", "segmentator_ref_O2")
        if os.path.exists(ref_bin):                  # the unmodified reference CLI in a child process (its stdout must not reach ours)
            with tempfile.TemporaryDirectory() as d:
                p = os.path.join(d, "m.ply"); synth.write_ply(p, xyz, tri)
                t0 = time.perf_counter(); r = subprocess.run([ref_bin, p], capture_output=True, text=True); rec["cpu_reference_s"] = time.perf_counter() - t0
                rec["cpu_reference_kind"] = "unmodified reference CLI (load + segment + segs.json), -O2, 1 thread"
                if r.returncode == 0:
                    with open(os.path.join(d, "m.0.010000.segs.json")) as fh:
                        rec["bit_identical_to_reference"] = bool((np.array(json.load(fh)["segIndices"]) == seg).all())
                ref0 = os.path.join(ROOT, "oracle", "_ref", "segmentator_ref")
                if os.path.exists(ref0):            # the reference's own Makefile flags (-std=c++11, i.e. -O0; Segmentator/Makefile:1-5)
                    t0 = time.perf_counter(); subprocess.run([ref0, p], capture_output=True, text=True); rec["cpu_reference_O0_s"] = time.perf_counter() - t0
                t0 = time.perf_counter(); r2 = subprocess.run([os.path.join(ROOT, "scannet_b200", "bin", "segmentator"), p], capture_output=True, text=True)
                rec["gpu_cli_s"] = time.perf_counter() - t0
                # the same mesh 8 times in ONE process (segmentator --batch): the CUDA context is paid once
                lst = os.path.join(d, "list.txt")
                paths = []
                for q in range(8):
                    pq = os.path.join(d, f"m{q}.ply"); shutil.copy(p, pq); paths.append(pq)
                with open(lst, "w") as fh:
                    fh.write("\n".join(paths) + "\n")
                t0 = time.perf_counter(); r3 = subprocess.run([os.path.join(ROOT, "scannet_b200", "bin", "segmentator"), "--batch", lst], capture_output=True, text=True)
                rec["gpu_cli_batch8_s_per_mesh"] = (time.perf_counter() - t0) / 8 if r3.returncode == 0 else None
        out[name] = rec
    return out


def sens_bench(n_frames=120):
    """SensReader decode throughput (R3/R4) vs the compiled reference, 1 thread, and the decode-inclusive `fuse` CLI
    (.sens -> TSDF -> marching cubes -> PLY) on a synthetic 640x480 zlib-depth stream."""
    import ctypes as C
    import tempfile
    from scannet_b200 import synth
    from scannet_b200.sens import SensFile
    out = {}
    ref_so_path = os.path.join(ROOT, "oracle", "_ref", "libref_sens.so")
    with tempfile.TemporaryDirectory() as d:
        sc, P = scene_poses(n_frames, 3, 1000)
        D = np.stack([sc.render(P[i], noise_mm=1.0, frame_seed=i)[0] for i in range(n_frames)])
        p = os.path.join(d, "s.sens")
        synth.write_sens(p, D, None, P, sc.intrinsics(), depth_comp=1, color_comp=0)
        s = SensFile(p)
        t0 = time.perf_counter()
        for i in range(n_frames):
            s.depth(i)
        out["depth_decode_fps_1thread"] = n_frames / (time.perf_counter() - t0)
        # the same frames inflated on the GPU, one warp per frame; 8 passes over the file's streams in one launch (960 frames)
        try:
            import ctypes as C2
            import torch
            from scannet_b200 import sens as _sens
            from scannet_b200._lib import check as _check, lib as _lib
            pay = []
            for i in range(n_frames):
                cp = C2.c_void_p(); dp = C2.c_void_p(); db = C2.c_uint64()
                _check(_lib().scn_sens_frame_payload(s._h, C2.c_uint64(i), C2.byref(cp), C2.byref(dp)))
                _check(_lib().scn_sens_frame_meta(s._h, C2.c_uint64(i), None, None, None, None, C2.byref(db)))
                pay.append(C2.string_at(dp.value, db.value))
            res = {}
            for reps in (4, 8, 32):                                                           # 480, 960 and 3840 frames in one launch
                streams = pay * reps
                dout = torch.empty((len(streams), H, W), dtype=torch.int16, device="cuda")
                _sens.inflate_batch_device(streams[:16], W * H * 2, dout.data_ptr())        # warm-up (staging buffers, module load)
                _sens.inflate_batch_device(streams, W * H * 2, dout.data_ptr())
                t0 = time.perf_counter(); _sens.inflate_batch_device(streams, W * H * 2, dout.data_ptr()); dt = time.perf_counter() - t0
                ok = bool((dout[-1].cpu().numpy().view(np.uint16) == D[-1]).all() and (dout[0].cpu().numpy().view(np.uint16) == D[0]).all())
                pk, kms, ring, _n = _sens.inflate_last_timings()
                res[f"{len(streams)}_frames"] = {"fps_incl_pack_and_h2d": len(streams) / dt, "ms": dt * 1e3, "kernel_ms": kms, "kernel_only_fps": len(streams) / (kms * 1e-3) if kms else None,
                                                 "host_pack_and_upload_issue_ms": pk * 1e3, "window": "shared-memory ring" if ring else "HBM (L2)", "identical_to_host_decode": ok}
                del dout
            res["compressed_bytes_per_frame"] = int(sum(len(b) for b in pay) / len(pay))
            res["deflate_block_type"] = "dynamic Huffman (zlib level 6)"
            out["depth_decode_gpu"] = res
            dout = None
            del dout
        except Exception as e:                                                                 # a side measurement must not take the bench line down
            out["depth_decode_gpu"] = {"error": repr(e)}
        ref_so = os.path.join(ROOT, "oracle", "_ref", "libref_sens.so")
        if os.path.exists(ref_so):
            L = C.CDLL(ref_so); L.ref_sens_open.restype = C.c_void_p; L.ref_sens_open.argtypes = [C.c_char_p]
            L.ref_sens_depth.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
            r = L.ref_sens_open(p.encode()); buf = np.zeros((H, W), np.uint16)
            t0 = time.perf_counter()
            for i in range(n_frames):
                L.ref_sens_depth(r, i, buf.ctypes.data)
            out["reference_depth_decode_fps_1thread"] = n_frames / (time.perf_counter() - t0)
        # colour (R4): JPEG 640x480 and 1296x968, host decoder 1 thread vs reference stb vs device decoder
        try:
            import cv2
            import torch
            from scannet_b200 import sens as _sens2
            col = {}
            for (cw, chh), reps in (((640, 480), 8), ((1296, 968), 4)):
                imgs = []
                yy, xx = np.mgrid[0:chh, 0:cw]
                for i in range(24):
                    im = np.stack([(xx * 255 // cw + 3 * i) % 256, (yy * 255 // chh + 5 * i) % 256, ((xx + yy) // 3 + 7 * i) % 256], -1).astype(np.uint8)
                    im = cv2.GaussianBlur(im, (0, 0), 1.5)
                    ok, buf = cv2.imencode(".jpg", im, [int(cv2.IMWRITE_JPEG_QUALITY), 85]); imgs.append(buf.tobytes())
                pj = os.path.join(d, f"c{cw}.sens")
                Dz = np.full((24, 8, 8), 1000, np.uint16); Pz = np.tile(np.eye(4, dtype=np.float32), (24, 1, 1)); it = iter(imgs)
                synth.write_sens(pj, Dz, np.zeros((24, chh, cw, 3), np.uint8), Pz, np.eye(4, dtype=np.float32), depth_comp=0, color_comp=2, jpeg_encoder=lambda x: next(it))
                sj = SensFile(pj)
                t0 = time.perf_counter()
                for i in range(24):
                    sj.color(i)
                rec = {"jpeg_bytes_per_frame": int(sum(len(b) for b in imgs) / 24), "host_decode_fps_1thread": 24 / (time.perf_counter() - t0)}
                if os.path.exists(ref_so_path):
                    Lr = C.CDLL(ref_so_path); Lr.ref_sens_open.restype = C.c_void_p; Lr.ref_sens_open.argtypes = [C.c_char_p]
                    Lr.ref_sens_color.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
                    rr = Lr.ref_sens_open(pj.encode()); bufc = np.zeros((chh, cw, 3), np.uint8)
                    t0 = time.perf_counter()
                    for i in range(24):
                        Lr.ref_sens_color(rr, i, bufc.ctypes.data)
                    rec["reference_stb_decode_fps_1thread"] = 24 / (time.perf_counter() - t0)
                jp = imgs * (reps * 10)
                dout = torch.empty((len(jp), chh, cw, 3), dtype=torch.uint8, device="cuda")
                _sens2.jpeg_decode_batch_device(jp[:24], cw, chh, dout.data_ptr())
                t0 = time.perf_counter(); k = _sens2.jpeg_decode_batch_device(jp, cw, chh, dout.data_ptr()); dt = time.perf_counter() - t0
                okc = bool((dout[-1].cpu().numpy() == sj.color(23)).all())
                hs, ems, cms = _sens2.jpeg_last_timings()
                rec["device"] = {"frames": len(jp), "decoded_on_device": k, "fps_incl_parse_pack_h2d": len(jp) / dt, "ms": dt * 1e3, "entropy_idct_kernel_ms": ems, "colour_kernel_ms": cms,
                                 "kernels_only_fps": len(jp) / ((ems + cms) * 1e-3) if ems else None, "host_parse_pack_upload_issue_ms": hs * 1e3, "identical_to_host_decode": okc}
                col[f"{cw}x{chh}"] = rec
                del dout
            out["color_decode"] = col
        except Exception as e:
            out["color_decode"] = {"error": repr(e)}
        prm = os.path.join(d, "p.txt")
        with open(prm, "w") as fh:
            fh.write("s_SDFVoxelSize = 0.004f;\ns_SDFTruncation = 0.02f;\ns_SDFTruncationScale = 0.01f;\n")
        t0 = time.perf_counter()
        r = subprocess.run([os.path.join(ROOT, "scannet_b200", "bin", "fuse"), prm, p], capture_output=True, text=True)
        out["fuse_cli_wall_s"] = time.perf_counter() - t0
        out["fuse_cli_stdout"] = [ln for ln in r.stdout.splitlines() if ln.startswith(("integrated", "mesh written"))]
        r = subprocess.run([os.path.join(ROOT, "scannet_b200", "bin", "fuse"), prm, p, os.path.join(d, "g.ply")], capture_output=True, text=True,
                           env=dict(os.environ, SCN_FUSE_DECODE="gpu"))
        out["fuse_cli_gpu_decode_stdout"] = [ln for ln in r.stdout.splitlines() if ln.startswith(("integrated", "depth decode"))]
    return out


# ----------------------------------------------------------------------------- decode-inclusive pipeline (configs[2])
def make_sens_file(path, n_frames, seed, device, color_wh=(1296, 968), with_color=True, threads=None, chunk=128):
    """A synthetic scan as a .sens file: 640x480 zlib depth (+ 1296x968 JPEG colour, ScannerApp/README.md:20-23) of the box-room
    scene along one camera loop.  Rendered on the device with torch, compressed by a host thread pool (zlib level 6, JPEG q85 —
    both release the GIL).  Returns (bytes written, seconds)."""
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    import cv2
    import torch
    from scannet_b200 import synth
    t0 = time.perf_counter()
    threads = threads or min(64, os.cpu_count() or 1)
    sc, P = scene_poses(n_frames, seed, n_frames)
    CW, CH = color_wh
    scc = synth.BoxRoomScene(size=(6.0, 5.0, 3.0), seed=seed, width=CW, height=CH, fx=synth.FX * CW / W, fy=synth.FY * CH / H,
                             cx=(synth.CX + 0.5) * CW / W - 0.5, cy=(synth.CY + 0.5) * CH / H - 0.5)
    Kc = scc.intrinsics()

    def enc(args):
        d, c = args
        ok, buf = (True, None) if c is None else cv2.imencode(".jpg", c, [int(cv2.IMWRITE_JPEG_QUALITY), 85])
        return (b"" if c is None else buf.tobytes()), zlib.compress(d.tobytes(), 6)

    with synth.SensWriter(path, n_frames, (W, H), (CW, CH) if with_color else (0, 0), sc.intrinsics(), Kc if with_color else None,
                          color_comp=2 if with_color else 0) as wr, ThreadPoolExecutor(threads) as ex:
        for s0 in range(0, n_frames, chunk):
            Pc = P[s0:s0 + chunk]
            d = render_depth_torch(sc, Pc, device).cpu().numpy().view(np.uint16)
            if with_color:
                dc = render_depth_torch(scc, Pc, device).to(torch.float32)                   # smooth shading of the same geometry at colour resolution
                col = torch.stack((128 + 100 * torch.sin(dc * 0.004), 128 + 100 * torch.sin(dc * 0.0023 + 1.0), 128 + 100 * torch.cos(dc * 0.0011)), -1)
                col = col.clamp(0, 255).to(torch.uint8).cpu().numpy()
                items = [(d[i], col[i]) for i in range(len(Pc))]
            else:
                items = [(d[i], None) for i in range(len(Pc))]
            for i, (cb, db) in enumerate(ex.map(enc, items)):
                wr.add(cb if with_color else b"", db, Pc[i])
    return os.path.getsize(path), time.perf_counter() - t0


def pipeline_bench(args, device):
    """BASELINE.json configs[2] stand-in: a 5,578-frame scan (1296x968 JPEG colour + 640x480 zlib depth) through the product
    driver scn_fuse_scene: compressed payloads -> GPU inflate + GPU JPEG -> hashed 4 mm TSDF -> marching cubes -> PLY."""
    import tempfile
    from scannet_b200 import fuse as sfuse
    out = {}
    with tempfile.TemporaryDirectory(dir=os.environ.get("SCN_BENCH_TMP")) as d:
        p = os.path.join(d, "scene.sens")
        nbytes, gen_s = make_sens_file(p, args.c3_frames, 7, device)
        out["input"] = {"frames": args.c3_frames, "depth": "640x480 u16 zlib-6", "colour": "1296x968 JPEG q85 4:2:0", "file_gb": round(nbytes / 1e9, 3),
                        "generation_s": round(gen_s, 1), "note": "synthetic stand-in for scene0000_00 (licence-gated, SURVEY.md §8d)"}
        for mode in ("gpu", "host"):
            rep = sfuse.fuse_scene(p, os.path.join(d, f"mesh_{mode}.ply"), max_blocks=1 << 22, hash_slots=1 << 24, decode_mode=mode)
            out[mode + "_decode"] = rep
        out["meshes_identical"] = open(os.path.join(d, "mesh_gpu.ply"), "rb").read() == open(os.path.join(d, "mesh_host.ply"), "rb").read()
    return out


def file_to_tsdf(args, device, rank, world, grp):
    """configs[1]/[3] decode-inclusive: every rank fuses its own 1000-frame .sens (depth zlib + 640x480 JPEG colour off) from file
    through scn_fuse_scene; the job's rate = all frames / max over ranks of the wall time (barrier before the start)."""
    import tempfile
    from scannet_b200 import fuse as sfuse
    with tempfile.TemporaryDirectory(dir=os.environ.get("SCN_BENCH_TMP")) as d:
        p = os.path.join(d, f"scene{rank}.sens")
        make_sens_file(p, args.scene_frames, 100 + rank, device, with_color=False, threads=max(4, (os.cpu_count() or 8) // max(world, 1)))
        sfuse.fuse_scene(p, None, decode_mode="gpu", device=device.index or 0)                 # warm-up: context, staging buffers, module load
        grp.barrier()
        t0 = time.perf_counter()
        rep = sfuse.fuse_scene(p, None, decode_mode="gpu", device=device.index or 0)
        dt = time.perf_counter() - t0
        frames, ms = grp.reduce_throughput(rep["frames_integrated"], dt * 1e3)
        res = {"value": frames / (ms / 1e3), "unit": UNIT, "frames": frames, "wall_s_max_over_ranks": ms / 1e3,
               "what": "file (.sens, zlib depth) -> GPU inflate -> TSDF, one scene per GPU, no mesh; includes opening + parsing the file and creating the volume",
               "rank0": rep}
        # the product multi-scene driver: every rank hands 8 scenes (the same file) to scn_fuse_many on its own GPU; the worker keeps
        # its volume and frame buffers from scene to scene
        dev = device.index or 0
        sfuse.fuse_many([p] * 2, None, devices=(dev,), decode_mode="gpu")
        grp.barrier()
        t0 = time.perf_counter()
        reps = sfuse.fuse_many([p] * 8, None, devices=(dev,), decode_mode="gpu")
        dt = time.perf_counter() - t0
        frames, ms = grp.reduce_throughput(sum(r["frames_integrated"] for r in reps), dt * 1e3)
        res["many"] = {"value": frames / (ms / 1e3), "unit": UNIT, "frames": frames, "scenes_per_gpu": 8, "wall_s_max_over_ranks": ms / 1e3,
                       "what": "scn_fuse_many: 8 scenes per GPU back to back (file -> GPU inflate -> TSDF), volume and frame buffers reused",
                       "rank0_scene_fuse_s": [round(r["fuse_s"], 4) for r in reps], "rank0_scene_total_s": [round(r["total_s"], 4) for r in reps],
                       "volume_reused": [r["volume_reused"] for r in reps]}
    return res


# ----------------------------------------------------------------------------- output dump
DUMP_BYTES = 64_000_000


def dump_outputs(d, vol):
    """Writes what the last timed step left in the volume, i.e. its last scene (the step resets the volume before each scene):
    the volume's counters, every allocated block's coordinates (sorted), and sdf / weight / colour of the voxels of a fixed
    seeded sample of those blocks (all of them when they fit), float32 / float64 .npy files of at most DUMP_BYTES in all."""
    os.makedirs(d, exist_ok=True)
    st = vol.stats()
    xyz, vox = vol.download_blocks()
    n = len(xyz)
    per_block = 512 * 5 * 4 + 8                                  # sdf, weight, r, g, b as float32 + the block's index
    k = min(n, (DUMP_BYTES - 12 * n - (1 << 16)) // per_block)
    pick = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False)) if k < n else np.arange(n)
    v = vox[pick]
    out = {"stats": np.array([st.frames_integrated, st.frames_skipped, st.blocks_allocated, st.voxels_updated, st.blocks_visited], np.float64),
           "block_xyz": xyz.astype(np.float32), "sample_block_index": pick.astype(np.float64),
           "sample_sdf": v["sdf"].astype(np.float32), "sample_weight": v["w"].astype(np.float32),
           "sample_rgb": np.stack([v["r"], v["g"], v["b"]], -1).astype(np.float32)}
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), a)
    return {"dir": d, "blocks": n, "sampled_blocks": int(k), "bytes": int(sum(a.nbytes for a in out.values()))}


# ----------------------------------------------------------------------------- GPU arm
def load_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "latest_traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames-per-step", type=int, default=4000, help="rounded down to whole 1000-frame scenes (configs[1])")
    ap.add_argument("--scene-frames", type=int, default=SCENE_FRAMES, help="frames per synthetic scene (1000 = configs[1]; smaller only for profiler runs)")
    ap.add_argument("--batch", type=int, default=32, help="frames fused per block residency (scn_tsdf_params.batch_frames)")
    ap.add_argument("--loop", type=int, default=1000, help="frames per camera loop of the synthetic trajectory")
    ap.add_argument("--cpu-frames", type=int, default=24, help="bounded CPU sample: frames per reference step")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--color", action="store_true", help="also fuse colour")
    ap.add_argument("--no-seg", action="store_true", help="skip the Segmentator / SensReader side sections")
    ap.add_argument("--no-seg-c5", action="store_true", help="skip the 2M-vertex Segmentator case")
    ap.add_argument("--tma-kernel", action="store_true", help="force the cp.async.bulk staged integrate kernel (SCN_TSDF_KERNEL_TMA)")
    ap.add_argument("--column-kernel", action="store_true", help="force the register-resident column kernel (SCN_TSDF_KERNEL_COLUMN)")
    ap.add_argument("--c3-frames", type=int, default=5578, help="frames of the configs[2] stand-in scan in the pipeline side section (0 = skip)")
    ap.add_argument("--parity-frames", type=int, default=64, help="frames of the in-bench parity check against the oracle (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the volume the last timed step computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    from scannet_b200 import dist as sdist
    from scannet_b200 import tsdf

    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the single JSON line
    rank, world, local = sdist.env_rank()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    grp = sdist.Group("nccl", dev)

    S, Wm = args.steps, args.warmup
    scene_frames = args.scene_frames
    n_sc = max(1, args.frames_per_step // scene_frames)
    F = n_sc * scene_frames
    frame_bytes = W * H * 2
    rgb_bytes = W * H * 3
    # every rank owns its own scenes (different sphere layouts per seed, same room size and camera loop, so the per-GPU work is
    # the same to within a few percent); every step replays them from an empty volume, so all steps do identical work
    scenes = []
    for j in range(n_sc):
        sc, P = scene_poses(scene_frames, sdist.scene_seed_for_rank(rank) * 16 + j, args.loop)
        d_depth = render_depth_torch(sc, P, dev)                                  # [1000,H,W] int16 (u16 bits), HBM resident
        h_depth = torch.empty(d_depth.shape, dtype=torch.int16, pin_memory=True)
        h_depth.copy_(d_depth)
        d_rgb = h_rgb = None
        if args.color:                                                             # synthetic colour registered to depth: [N,H,W,3] u8
            dd = d_depth.to(torch.int32) & 0xFFFF
            d_rgb = torch.stack(((dd >> 4) & 255, (dd >> 2) & 255, dd & 255), dim=-1).to(torch.uint8).contiguous()
            h_rgb = torch.empty(d_rgb.shape, dtype=torch.uint8, pin_memory=True)
            h_rgb.copy_(d_rgb)
            del dd
        scenes.append({"sc": sc, "P": P, "K": sc.intrinsics(), "d": d_depth, "h": h_depth, "dc": d_rgb, "hc": h_rgb})
    torch.cuda.synchronize()

    def make_volume(flags=0):
        p = tsdf.default_params(batch_frames=args.batch, max_blocks=1 << 20, hash_slots=1 << 22,
                                flags=flags | (tsdf.KERNEL_TMA if args.tma_kernel else 0) |
                                (tsdf.KERNEL_COLUMN if args.column_kernel else 0))
        return tsdf.TsdfVolume(p, device=local, stream=torch.cuda.current_stream().cuda_stream)

    barrier = grp.barrier

    def timed(fn_step):
        """W warm-up steps, then exactly S steps bracketed by barrier+sync, CUDA events on the launch stream."""
        for s in range(Wm):
            fn_step(s)
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(Wm, Wm + S):
            fn_step(s)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        return grp.reduce_throughput(S * F, ms)       # (frames over all ranks, max ms over ranks)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()

    # ---- pass 1: device-resident inputs ------------------------------------------------------
    vol = make_volume()
    acc = {"nu": 0, "nb": 0, "blocks": 0, "launches": 0, "collect": True, "prof": False}

    def step_dev(s):
        if s == Wm and not acc["prof"]:
            vol.sync(); vol.profile(True); acc["prof"] = True      # kernel timing events: timed steps only
        for sc in scenes:
            vol.reset()                                              # empty volume (clears only the blocks the last scene used)
            vol.integrate_device(scene_frames, sc["d"].data_ptr(), sc["dc"].data_ptr() if sc["dc"] is not None else None, sc["P"], sc["K"])
            if acc["collect"]:                                       # first (warm-up) step only: per-step counters, identical in every step
                vol.sync(); st = vol.stats()
                acc["nu"] += st.voxels_updated; acc["nb"] += st.blocks_visited; acc["blocks"] += st.blocks_allocated
                acc["launches"] += st.kernel_launches + 1            # + the reset's block-clearing kernel
        acc["collect"] = False

    if Wm < 1:
        step_dev(-1)
    frames_all, ms_dev = timed(step_dev)
    vol.sync()
    alloc_ms, integ_ms, n_batches, _ = vol.kernel_times()
    dumped = dump_outputs(args.dump_outputs, vol) if args.dump_outputs and rank == 0 else None
    vol.close()

    # ---- pass 2: end to end from pinned host memory -------------------------------------------
    vol2 = make_volume()

    def step_e2e(s):
        for sc in scenes:
            vol2.reset()
            vol2.integrate_batch_ptr(scene_frames, sc["h"].data_ptr(), sc["hc"].data_ptr() if sc["hc"] is not None else None, sc["P"], sc["K"])
            vol2.stats()                                            # D2H read of the scene's result (counters)

    frames_all2, ms_e2e = timed(step_e2e)
    vol2.sync()
    vol2.close()
    clocks = sampler.stop() if sampler else None
    # ---- decode-inclusive: .sens file -> TSDF through the product driver, one scene per rank ------------------------------
    f2t = None
    if not args.no_seg:
        try:
            f2t = file_to_tsdf(args, dev, rank, world, grp)
        except Exception as e:
            f2t = {"error": repr(e)}

    # ---- in-bench parity check: the first frames of scene 0 through the same entry point, bit for bit against the oracle ----
    parity = None
    if rank == 0 and args.parity_frames > 0:
        import hashlib
        import oracle_bindings as ob
        npar = (args.parity_frames // args.batch) * args.batch or args.parity_frames
        sc0 = scenes[0]
        v3 = make_volume()
        v3.integrate_device(npar, sc0["d"].data_ptr(), sc0["dc"].data_ptr() if sc0["dc"] is not None else None, sc0["P"][:npar], sc0["K"])
        v3.sync()
        gx, gv = v3.download_blocks(); st3 = v3.stats(); v3.close()
        _omp_env()
        o = ob.OracleTsdf(bench_params(), threads=min(os.cpu_count() or 1, 32))
        Dh = sc0["h"][:npar].numpy().view(np.uint16)
        Ch = sc0["hc"][:npar].numpy() if sc0["hc"] is not None else None
        for i in range(npar):
            o.integrate(Dh[i], None if Ch is None else Ch[i], sc0["P"][i], sc0["K"])
        ox, ov = o.export(); oc = o.counters(); o.close()
        same = bool(gx.shape == ox.shape and (gx == ox).all() and gv.tobytes() == ov.tobytes()
                    and st3.voxels_updated == oc["total_updated"] and st3.blocks_visited == oc["total_touched"])
        parity = {"frames": npar, "entry": "scn_tsdf_integrate_device", "bit_identical_to_oracle": same, "blocks": int(len(gx)),
                  "voxel_updates": int(st3.voxels_updated),
                  "sha256_gpu": hashlib.sha256(gx.tobytes() + gv.tobytes()).hexdigest()[:16],
                  "sha256_oracle": hashlib.sha256(ox.tobytes() + ov.tobytes()).hexdigest()[:16],
                  "oracle": "oracle/tsdf_oracle.c (own spec v1.1 — parity unpinned: the reference has no TSDF source)"}

    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        value = frames_all / (ms_dev / 1e3)
        e2e = frames_all2 / (ms_e2e / 1e3)
        alg_integrate = 16.0 * (acc["nu"] + acc["nb"]) * S          # bytes, integrate kernel, timed steps (this rank)
        per_launch_bytes = alg_integrate / max(n_batches, 1)
        per_launch_ms = integ_ms / max(n_batches, 1)
        achieved = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else 0.0
        tj = load_traffic()
        kname = tj.get("integrate_kernel", "k_integrate_col")
        traffic = tj.get("dram_bytes_per_launch", {}).get(kname) if args.batch == tj.get("batch") else None
        dram_gbs = traffic / (per_launch_ms * 1e-3) / 1e9 if traffic and per_launch_ms > 0 else None
        cfg = make_config(args, world)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": S, "warmup": Wm,
            "ms_per_step": ms_dev / S, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "timed_region_s": ms_dev / 1e3, "frames_timed": S * F, "blocks_allocated_per_step": int(acc["blocks"]),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": F * (frame_bytes + (rgb_bytes if args.color else 0)),
                    "d2h_bytes_per_step": 64 * n_sc, "ms_per_step": ms_e2e / S, "timed_region_s": ms_e2e / 1e3},
            "gpu_launches": int(acc["launches"]) * S,
            "roofline": {"bound": "issue", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": f"profiles/latest_traffic.json ({tj.get('tag')}: ncu dram__bytes read+write per launch, batch {tj.get('batch')})" if traffic else None,
                         "dram_gbs": dram_gbs, "dram_frac": dram_gbs / peak if dram_gbs else None,
                         "issue_active": tj.get("issue_active", {}).get(kname),
                         "warp_inst_per_voxel_frame": tj.get("thread_inst_per_voxel_frame", {}).get(kname),
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": per_launch_bytes, "avg_launch_ms": per_launch_ms,
                         "launches": int(n_batches),
                         "kernel_share_of_step": integ_ms / ms_dev if ms_dev else None,
                         "alloc_kernel_ms_total": alloc_ms, "integrate_kernel_ms_total": integ_ms,
                         "note": "achieved/frac use SURVEY.md §8d algorithmic bytes (16 B per voxel update + 16 B per block visit, per frame) over the "
                                 "integrate kernel's event-timed duration. Fusing K frames per block residency makes real DRAM traffic (dram_gbs, from "
                                 "the ncu capture) ~10x lower than that figure, so frac can exceed 1: the kernel is bound by instruction issue "
                                 "(issue_active), not by HBM; the two kernels of consecutive batches overlap, so their times sum to more than the step"},
            "parity_check": parity,
            "dumped_outputs": dumped,
            "file_to_tsdf": f2t,
            "clocks": clocks,
        }
        if world == 1 and not args.no_seg:          # side sections first: the CPU arm below perturbs host-side timings measured after it
            try:
                line["segmentator"] = seg_bench(not args.no_seg_c5)
            except Exception as e:          # the side benchmarks must never take the headline line down
                line["segmentator"] = {"error": repr(e)}
            try:
                line["sens"] = sens_bench()
            except Exception as e:
                line["sens"] = {"error": repr(e)}
            if args.c3_frames > 0:
                try:
                    line["pipeline_c3"] = pipeline_bench(args, dev)
                except Exception as e:
                    line["pipeline_c3"] = {"error": repr(e)}
        if not args.no_cpu and world == 1:          # CPU baseline: rank 0 at N=1 only
            line["cpu_baseline"], _ = cpu_arm(args, steps=1, warmup=0)
        emit(line)
    grp.close()


if __name__ == "__main__":
    main()
