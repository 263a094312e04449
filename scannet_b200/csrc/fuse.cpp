// `fuse` — the reconstruction stage contract of the reference pipeline in library form:
//   <exe> <params.txt> [<params2.txt>] <file.sens> [out.ply]        (Server/scan_processor.py:27-35,123-138)
//   <exe> --gpus N <params.txt> ... <a.sens> <b.sens> ...           one scene per GPU at a time (Server/process.py:75 serialises
//                                                                   one scan per GPU; here N scans run on N GPUs, SURVEY.md §8e)
// Reads the .sens stream (SensReader), fuses every frame that has a valid pose into the hashed TSDF volume (poses come from
// the file: camera tracking / bundle adjustment is not part of this path), extracts the surface with marching cubes and
// writes `<base>_vh.ply` in the VCGLIB layout the `segment` stage reads (Server/config/scan_stages.json:33-37).
//
// Decode.  Both modes run one chunk pipeline: the frames with a valid pose are planned in chunks, and decode lanes fill
// double-buffered frame arrays one chunk ahead of the integrator.  "gpu" (default for zlib or raw depth): the COMPRESSED payloads
// are decoded in HBM — depth by the inflate kernel (csrc/inflate.cu), JPEG colour by csrc/jpeg_gpu.cu, which samples only the
// colour pixels the depth image needs; raw depth is uploaded as it is, raw / PNG colour decoded by a host thread pool.  "host"
// (SCN_FUSE_DECODE=host): a host thread pool decodes depth and colour into pinned memory; the GPU decoders are tested against it.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "scn_common.h"
#include "stage_pool.h"

namespace {

// Persistent worker pool: run(fn) executes fn() on every worker and on the caller, and returns when all are done
// (spawning 64 threads per 128-frame chunk cost ~3 ms of a ~10 ms chunk).
class Pool {
 public:
  explicit Pool(unsigned workers) { for (unsigned i = 0; i < workers; ++i) th_.emplace_back([this]() { loop(); }); }
  ~Pool() { { std::lock_guard<std::mutex> l(m_); stop_ = true; ++gen_; } cv_.notify_all(); for (auto& t : th_) t.join(); }
  void run(const std::function<void()>& fn) {
    { std::lock_guard<std::mutex> l(m_); fn_ = &fn; pending_ = (unsigned)th_.size(); ++gen_; }
    cv_.notify_all();
    fn();
    std::unique_lock<std::mutex> l(m_); done_.wait(l, [this]() { return pending_ == 0; });
  }
 private:
  void loop() {
    unsigned long seen = 0;
    for (;;) {
      const std::function<void()>* fn;
      { std::unique_lock<std::mutex> l(m_); cv_.wait(l, [&]() { return gen_ != seen; }); seen = gen_; if (stop_) return; fn = fn_; }
      (*fn)();
      { std::lock_guard<std::mutex> l(m_); if (--pending_ == 0) done_.notify_one(); }
    }
  }
  std::vector<std::thread> th_; std::mutex m_; std::condition_variable cv_, done_;
  const std::function<void()>* fn_ = nullptr; unsigned pending_ = 0; unsigned long gen_ = 0; bool stop_ = false;
};

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// colour pixel for every depth pixel: K_c * K_d^-1 * (x, y, 1), nearest (sensorData.h:1577-1586 with identity extrinsics)
void build_color_lut(const scn_sens_info_t& in, std::vector<int32_t>& lut) {
  const uint32_t W = in.depth_width, H = in.depth_height;
  lut.resize((size_t)W * H);
  const float fxd = in.depth_intrinsic[0], cxd = in.depth_intrinsic[2], fyd = in.depth_intrinsic[5], cyd = in.depth_intrinsic[6];
  const float fxc = in.color_intrinsic[0], cxc = in.color_intrinsic[2], fyc = in.color_intrinsic[5], cyc = in.color_intrinsic[6];
  for (uint32_t y = 0; y < H; ++y) for (uint32_t x = 0; x < W; ++x) {
    const float u = ((float)x - cxd) / fxd * fxc + cxc, v = ((float)y - cyd) / fyd * fyc + cyc;
    const long cx = lrintf(u), cy = lrintf(v);
    lut[(size_t)y * W + x] = (cx >= 0 && cy >= 0 && cx < (long)in.color_width && cy < (long)in.color_height) ? (int32_t)(cy * in.color_width + cx) : -1;
  }
}

// a decoded colour frame registered to the depth image: out[p] = col[lut[p]], black where lut[p] < 0
void register_color(const std::vector<int32_t>& lut, const uint8_t* col, uint8_t* out) {
  for (size_t p = 0; p < lut.size(); ++p) {
    const int32_t q = lut[p];
    if (q >= 0) { out[3 * p] = col[3 * (size_t)q]; out[3 * p + 1] = col[3 * (size_t)q + 1]; out[3 * p + 2] = col[3 * (size_t)q + 2]; }
    else out[3 * p] = out[3 * p + 1] = out[3 * p + 2] = 0;
  }
}

// decode(i, colour scratch of scratch_bytes) for the frames i < n of a chunk, on every thread of `pool`.  Stops at the first failure
// and returns its code; its text, thread-local to the worker that failed, is set again on the calling thread.
int decode_on_pool(Pool& pool, uint32_t n, size_t scratch_bytes, const std::function<int(uint32_t, uint8_t*)>& decode) {
  std::atomic<uint32_t> next{0}; std::atomic<int> rc{0}; std::mutex err_m; std::string err;
  pool.run([&]() {
    static thread_local std::vector<uint8_t> col;                               // kept per pool thread: no 1-4 MB allocation per chunk
    col.resize(scratch_bytes);
    for (uint32_t i; (i = next.fetch_add(1)) < n && !rc.load();)
      if (const int r = decode(i, col.data())) { std::lock_guard<std::mutex> l(err_m); if (!rc.load()) { err = scn_last_error(); rc.store(r); } }
  });
  return rc.load() ? scn::fail(rc.load(), "%s", err.c_str()) : SCN_OK;
}

// ---- one scene on one GPU ------------------------------------------------------------------------------------------------------
struct SceneJob {
  std::string sens_path, out_path;          // out_path empty = no mesh
  scn_tsdf_params params;                   // width / height / depth_shift are taken from the stream
  int device = 0;
  bool verbose = true;
  const char* decode_mode = nullptr;        // "gpu", "host" or null (automatic)
};

// The volume (16 GiB of voxel blocks with the CLI's defaults: cudaMalloc + first clear + cudaFree cost 0.15-0.4 s, as much as
// fusing a 5,578-frame scan; a reset clears only the used blocks in a few ms) is kept per device from one scene to the next - by
// the workers of scn_fuse_many and by consecutive scn_fuse_scene calls of a process alike; scn_release_cached_staging frees it.
struct VolSlot {
  int device = 0;
  scn_tsdf* vol = nullptr; scn_tsdf_params p;
  void release() { if (vol) scn_tsdf_destroy(vol); vol = nullptr; }
};
// The double-buffered frame arrays of the GPU-decode mode (3 GB at 1024-frame chunks with colour) come from a per-device pool
// like the decoders' staging: allocating and freeing them per scene cost up to 0.2 s (cudaFree synchronises the device).
struct FrameBufs {
  int device = 0;
  void* buf[4] = {nullptr, nullptr, nullptr, nullptr}; size_t cap[4] = {0, 0, 0, 0};       // depth x2, colour x2
  void* take(int i, size_t bytes) {
    if (bytes > cap[i]) { scn_device_free(buf[i]); buf[i] = scn_device_alloc(bytes); cap[i] = buf[i] ? bytes : 0; }
    return buf[i];
  }
  void release() { for (int i = 0; i < 4; ++i) { scn_device_free(buf[i]); buf[i] = nullptr; cap[i] = 0; } }
};
scn::StagePool<FrameBufs>& frame_pool() { static auto* p = new scn::StagePool<FrameBufs>(); return *p; }
scn::StagePool<VolSlot>& vol_pool() { static auto* p = new scn::StagePool<VolSlot>(); return *p; }

// Chunk c lists the frames of [c * chunk, (c + 1) * chunk) that have a valid pose: a frame without one is never decoded
// (sensorData.h:382), so a corrupt payload there cannot fail the run.
struct ChunkPlan {
  std::vector<uint64_t> frames; std::vector<float> poses;
  std::vector<const uint8_t*> src[2]; std::vector<uint64_t> len[2];        // compressed depth [0] and colour [1]: views into the stream
};

struct Scene {
  scn_sens* s = nullptr; scn_sens_info_t in; int device = 0;
  size_t px = 0; uint32_t chunk = 0;                       // depth pixels per frame, frames per chunk
  std::vector<int32_t> lut;                                // colour pixel of every depth pixel; empty = fused without colour
  std::vector<ChunkPlan> plan;
  uint16_t* depth[2] = {nullptr, nullptr}; uint8_t* rgb[2] = {nullptr, nullptr};   // the double-buffered frame arrays
};

// returns the number of frames without a pose
uint64_t plan_chunks(Scene& sc) {
  sc.plan.assign((sc.in.n_frames + sc.chunk - 1) / sc.chunk, ChunkPlan());
  uint64_t skipped = 0;
  for (uint64_t f = 0; f < sc.in.n_frames; ++f) {
    float T[16]; uint64_t cb = 0, db = 0; const uint8_t* cp = nullptr; const uint8_t* dp = nullptr;
    scn_sens_frame_meta(sc.s, f, T, nullptr, nullptr, &cb, &db); scn_sens_frame_payload(sc.s, f, &cp, &dp);
    if (T[0] == -INFINITY) { ++skipped; continue; }
    ChunkPlan& pl = sc.plan[f / sc.chunk];
    pl.frames.push_back(f); pl.poses.insert(pl.poses.end(), T, T + 16);
    pl.src[0].push_back(dp); pl.len[0].push_back(db); pl.src[1].push_back(cp); pl.len[1].push_back(cb);
  }
  return skipped;
}

// a decode lane fills its part (depth, colour or both) of a chunk's frames into buffer `b`; its time is added to *busy_s
struct Lane { std::function<int(const ChunkPlan& pl, int b)> fill; double* busy_s; };

// The pipeline of both decode modes.  Every lane runs on a thread of its own and fills chunk c into buffer c & 1 once
// c < consumed + 2; the integrator waits for every lane of chunk c, integrates it and waits for the GPU, after which buffer c & 1
// may be filled again.  The first failure stops every lane; its code is returned with its text.
int run_chunks(const Scene& sc, scn_tsdf* vol, const std::vector<Lane>& lanes, decltype(&scn_tsdf_integrate_device) integrate, scn_fuse_report_t& rep) {
  std::mutex m; std::condition_variable cv;
  std::vector<uint64_t> filled(lanes.size(), 0);                                // chunks each lane has finished
  uint64_t consumed = 0;                                                          // chunks whose buffers are free again
  int rc = SCN_OK; std::string err;                                               // the first failure
  auto failed = [&](int r) { { std::lock_guard<std::mutex> l(m); if (!rc) { rc = r; err = scn_last_error(); } } cv.notify_all(); };
  std::vector<std::thread> th;
  for (size_t k = 0; k < lanes.size(); ++k)
    th.emplace_back([&, k]() {
      scn_set_device(sc.device);
      for (uint64_t c = 0; c < sc.plan.size(); ++c) {
        { std::unique_lock<std::mutex> l(m); cv.wait(l, [&]() { return rc || c < consumed + 2; }); if (rc) return; }
        const double t = now_s();
        const int r = sc.plan[c].frames.empty() ? SCN_OK : lanes[k].fill(sc.plan[c], (int)(c & 1));
        *lanes[k].busy_s += now_s() - t;
        if (r) { failed(r); return; }
        { std::lock_guard<std::mutex> l(m); filled[k] = c + 1; } cv.notify_all();
      }
    });
  for (uint64_t c = 0; c < sc.plan.size(); ++c) {
    const double tw0 = now_s();
    { std::unique_lock<std::mutex> l(m); cv.wait(l, [&]() { return rc || *std::min_element(filled.begin(), filled.end()) > c; }); if (rc) break; }
    rep.decode_wait_s += now_s() - tw0;
    const ChunkPlan& pl = sc.plan[c];
    if (!pl.frames.empty()) {
      const double ti0 = now_s();
      int r = integrate(vol, (uint32_t)pl.frames.size(), sc.depth[c & 1], sc.rgb[c & 1], pl.poses.data(), sc.in.depth_intrinsic);
      if (!r) r = scn_tsdf_sync(vol);                                             // buffer c & 1 may be filled again now
      if (r) { failed(r); break; }
      rep.integrate_s += now_s() - ti0;
    }
    { std::lock_guard<std::mutex> l(m); consumed = c + 1; } cv.notify_all();
  }
  const double tt0 = now_s();
  for (std::thread& t : th) t.join();
  rep.teardown_s = now_s() - tt0;
  return rc ? scn::fail(rc, "%s", err.c_str()) : SCN_OK;
}

// GPU decode: the frame arrays live in HBM; a depth lane (inflate kernel, or one upload per raw frame) and a colour lane (device
// JPEG decoder, or for raw / PNG colour the host pool into a pinned chunk, registered to depth on the way, and one upload).  Host
// decode: the frame arrays live in pinned memory, filled by one lane whose host pool decodes each frame's depth and registered
// colour; scn_tsdf_integrate_batch uploads a chunk while the lane decodes the next one.
int fuse_chunks(Scene& sc, bool gpu, unsigned threads, scn_tsdf* vol, scn_fuse_report_t& rep) {
  const double t0 = now_s();
  const size_t CH = sc.chunk, px = sc.px, col_bytes = (size_t)sc.in.color_width * sc.in.color_height * 3;
  const bool use_color = !sc.lut.empty(), jpeg = sc.in.color_compression == 2;
  scn::StagePool<FrameBufs>::Lease fb(frame_pool());
  auto alloc = [&](int i, size_t bytes) { return gpu ? fb->take(i, bytes) : scn_host_alloc(bytes); };
  int32_t* d_lut = nullptr; void* st_d = nullptr; void* st_c = nullptr; uint8_t* h_rgb = nullptr; int rc = SCN_OK;
  for (int b = 0; b < 2 && !rc; ++b) {
    sc.depth[b] = (uint16_t*)alloc(b, CH * px * 2);
    if (use_color) sc.rgb[b] = (uint8_t*)alloc(2 + b, CH * px * 3);
    if (!sc.depth[b] || (use_color && !sc.rgb[b])) rc = SCN_ERR_CUDA;
  }
  if (!rc && gpu && use_color && jpeg) rc = (d_lut = (int32_t*)scn_device_alloc(px * 4)) ? scn_memcpy_h2d(d_lut, sc.lut.data(), px * 4, nullptr) : SCN_ERR_CUDA;
  if (!rc && gpu) rc = scn_stream_create(&st_d);
  if (!rc && gpu) rc = scn_stream_create(&st_c);
  rep.buffers_s = now_s() - t0;
  // the host decoders: of every frame in host mode, of raw / PNG colour in GPU mode
  Pool pool(!gpu ? threads - 1 : use_color && !jpeg ? std::max(1u, std::min(32u, std::thread::hardware_concurrency())) - 1 : 0);
  std::vector<Lane> lanes;
  if (!gpu) lanes.push_back({[&](const ChunkPlan& pl, int b) {                     // its time counts as depth decode
    return decode_on_pool(pool, (uint32_t)pl.frames.size(), use_color ? col_bytes : 0, [&](uint32_t i, uint8_t* col) {
      int q = scn_sens_frame_depth_u16(sc.s, pl.frames[i], sc.depth[b] + (size_t)i * px);
      if (!q && use_color && !(q = scn_sens_frame_color_rgb8(sc.s, pl.frames[i], col))) register_color(sc.lut, col, sc.rgb[b] + (size_t)i * px * 3);
      return q;
    });
  }, &rep.depth_decode_s});
  if (gpu) lanes.push_back({[&](const ChunkPlan& pl, int b) {
    const uint32_t n = (uint32_t)pl.frames.size();
    if (sc.in.depth_compression == 1) {
      const int r = scn_inflate_batch_device(pl.src[0].data(), pl.len[0].data(), n, (uint64_t)px * 2, sc.depth[b], st_d);
      double ps = 0, km = 0; scn_inflate_last_timings(&ps, &km, nullptr, nullptr);
      rep.depth_pack_s += ps; rep.depth_kernel_s += km * 1e-3;
      return r;
    }
    for (uint32_t i = 0; i < n; ++i)                                               // raw depth: uploaded as it is
      if (const int r = pl.len[0][i] < px * 2 ? scn::fail(SCN_ERR_FORMAT, "frame %llu: invalid data", (unsigned long long)pl.frames[i])
                                              : scn_memcpy_h2d(sc.depth[b] + (size_t)i * px, pl.src[0][i], px * 2, st_d)) return r;
    return SCN_OK;
  }, &rep.depth_decode_s});
  if (gpu && use_color && jpeg) lanes.push_back({[&](const ChunkPlan& pl, int b) {
    uint32_t k = 0; double hs = 0, em = 0, cm = 0;
    const int r = scn_jpeg_decode_batch_device(pl.src[1].data(), pl.len[1].data(), (uint32_t)pl.frames.size(), sc.in.color_width, sc.in.color_height,
                                               d_lut, (uint32_t)px, sc.rgb[b], st_c, &k);
    scn_jpeg_last_timings(&hs, &em, &cm);
    rep.color_frames_on_device += k; rep.color_host_s += hs; rep.color_entropy_s += em * 1e-3; rep.color_convert_s += cm * 1e-3;
    return r;
  }, &rep.color_decode_s});
  if (gpu && use_color && !jpeg) lanes.push_back({[&](const ChunkPlan& pl, int b) {
    const uint32_t n = (uint32_t)pl.frames.size();
    if (!h_rgb && !(h_rgb = (uint8_t*)scn_host_alloc(CH * px * 3))) return SCN_ERR_CUDA;
    const int r = decode_on_pool(pool, n, col_bytes, [&](uint32_t i, uint8_t* col) {
      const int q = scn_sens_frame_color_rgb8(sc.s, pl.frames[i], col);
      if (!q) register_color(sc.lut, col, h_rgb + (size_t)i * px * 3);
      return q;
    });
    return r ? r : scn_memcpy_h2d(sc.rgb[b], h_rgb, (size_t)n * px * 3, st_c);
  }, &rep.color_decode_s});
  if (!rc) rc = run_chunks(sc, vol, lanes, gpu ? scn_tsdf_integrate_device : scn_tsdf_integrate_batch, rep);
  const double tt0 = now_s();
  scn_device_free(d_lut); scn_stream_destroy(st_d); scn_stream_destroy(st_c); scn_host_free(h_rgb);
  if (!gpu) for (int b = 0; b < 2; ++b) { scn_host_free(sc.depth[b]); scn_host_free(sc.rgb[b]); }
  rep.teardown_s += now_s() - tt0;
  return rc;
}

// counters, marching cubes and the PLY
int finish(const SceneJob& job, scn_tsdf* vol, bool use_color, scn_fuse_report_t& rep) {
  scn_tsdf_stats_t st;
  if (const int rc = scn_tsdf_stats(vol, &st)) return rc;
  rep.frames_integrated = st.frames_integrated; rep.frames_skipped = st.frames_skipped + rep.frames_skipped_pose;
  rep.blocks_allocated = st.blocks_allocated; rep.voxels_updated = st.voxels_updated;
  if (job.verbose)
    printf("integrated %llu frames (%llu skipped: invalid pose) in %.3f s = %.1f frames/s incl. decode; %llu blocks, %llu voxel updates\n",
           (unsigned long long)rep.frames_integrated, (unsigned long long)rep.frames_skipped, rep.fuse_s, rep.frames_integrated / std::max(rep.fuse_s, 1e-9),
           (unsigned long long)st.blocks_allocated, (unsigned long long)st.voxels_updated);
  size_t used = 0, total = 0; if (!scn_device_mem_info(&used, &total)) rep.device_bytes_in_use = used;
  if (job.out_path.empty()) return SCN_OK;
  const double tm0 = now_s();
  float* xyz = nullptr; uint8_t* rgb = nullptr; uint32_t* tri = nullptr; uint64_t nV = 0, nF = 0;
  int rc = scn_tsdf_extract_mesh(vol, &xyz, &rgb, &tri, &nV, &nF);
  rep.mc_s = now_s() - tm0;
  if (!rc) rc = scn_mesh_save_ply(job.out_path.c_str(), xyz, use_color ? rgb : nullptr, nV, tri, nF);
  rep.ply_s = now_s() - tm0 - rep.mc_s;
  rep.mesh_vertices = nV; rep.mesh_faces = nF;
  if (!rc && job.verbose) printf("mesh written to %s with %llu vertices, %llu faces\n", job.out_path.c_str(), (unsigned long long)nV, (unsigned long long)nF);
  scn_free(xyz); scn_free(rgb); scn_free(tri);
  return rc;
}

// every failure of a scene reaches the caller with its own code, the .sens path in front of its text
int scene_error(const SceneJob& job, int rc) { return scn::fail(rc, "%s: %s", job.sens_path.c_str(), scn_last_error()); }

// setup -> plan -> run the chunks -> finish
int fuse_scene(const SceneJob& job, scn_fuse_report_t* rep_out) {
  scn_fuse_report_t rep; memset(&rep, 0, sizeof(rep));
  rep.device = job.device;
  const double t_begin = now_s();
  Scene sc; sc.device = job.device;
  int rc = scn_set_device(job.device);
  if (!rc) {
    std::thread warm([dev = job.device]() { scn_set_device(dev); scn_cuda_warmup(); });          // context creation overlaps reading the .sens file
    rc = scn_sens_open(job.sens_path.c_str(), &sc.s);
    warm.join();
  }
  if (rc) return scene_error(job, rc);
  const scn_sens_info_t& in = sc.in; scn_sens_info(sc.s, &sc.in);
  scn_tsdf_params p = job.params;
  p.width = in.depth_width; p.height = in.depth_height; p.depth_shift = in.depth_shift;   // integrate at the stream's depth resolution
  if (p.batch_frames == 0) p.batch_frames = 32;
  const bool use_color = in.color_compression <= 2 && in.color_width > 0 && in.color_height > 0;   // raw, PNG, JPEG (sensorData.h:600-616)
  if (job.verbose)
    printf("fusing %s: %llu frames %ux%u, voxel %.4f m, truncation %.3f+%.3f*d\n", job.sens_path.c_str(), (unsigned long long)in.n_frames, in.depth_width,
           in.depth_height, p.voxel_size, p.trunc_base, p.trunc_scale);
  scn::StagePool<VolSlot>::Lease vs(vol_pool());
  if (vs->vol && !memcmp(&vs->p, &p, sizeof(p))) { rep.volume_reused = 1; rc = scn_tsdf_reset(vs->vol); }   // same volume layout as the previous scene on this GPU
  else { vs->release(); vs->p = p; rc = scn_tsdf_create(&p, job.device, &vs->vol); }
  if (!rc) {
    sc.px = (size_t)in.depth_width * in.depth_height;
    if (use_color) build_color_lut(in, sc.lut);
    const bool gpu_decode = (in.depth_compression == 0 || in.depth_compression == 1) && !(job.decode_mode && !strcmp(job.decode_mode, "host"));
    if (job.verbose)
      printf("decode: %s\n", !gpu_decode ? "host thread pool" : (use_color && in.color_compression != 2) ? "GPU inflate (depth), host thread pool (raw / PNG colour)"
                                                                                        : "GPU inflate (depth) + GPU JPEG (colour), compressed payloads uploaded");
    rep.gpu_decode = gpu_decode ? 1 : 0;
    const double t0 = now_s();
    rep.setup_s = t0 - t_begin;
    // frames per chunk.  GPU: enough streams in flight for the one-warp-per-frame decoders.  Host: decode is the bottleneck of this
    // mode (one frame = ~2 ms inflate + ~1-3 ms JPEG on one core): up to 64 cores, two frames per thread.
    const char* ce = getenv("SCN_FUSE_CHUNK");
    const unsigned threads = std::max(1u, std::min(64u, std::thread::hardware_concurrency()));
    sc.chunk = gpu_decode ? (uint32_t)std::max(16, std::min(4096, ce ? atoi(ce) : 1024)) : std::max(32u, 2 * threads);
    rep.frames_skipped_pose = plan_chunks(sc);
    rc = fuse_chunks(sc, gpu_decode, threads, vs->vol, rep);
    rep.fuse_s = now_s() - t0;
    if (!rc) rc = finish(job, vs->vol, use_color, rep);
  }
  if (rc) vs->release();                                       // do not hand a volume of unknown state to the next scene
  scn_sens_close(sc.s);
  rep.total_s = now_s() - t_begin;
  if (rep_out) *rep_out = rep;
  return rc ? scene_error(job, rc) : SCN_OK;
}

std::string default_out(const std::string& sens_path) { return sens_path.substr(0, sens_path.size() - 5) + "_vh.ply"; }

}  // namespace

extern "C" {

void scn_fuse_release_staging_() { frame_pool().trim(); vol_pool().trim(); }
size_t scn_fuse_report_sizeof(void) { return sizeof(scn_fuse_report_t); }

int scn_fuse_scene(const char* sens_path, const char* out_ply, const scn_tsdf_params* params, int device, const char* decode_mode, scn_fuse_report_t* report) {
  if (!sens_path || !params) return scn::fail(SCN_ERR_ARG, "null argument");
  SceneJob j; j.sens_path = sens_path; j.out_path = out_ply ? out_ply : ""; j.params = *params; j.device = device; j.verbose = false; j.decode_mode = decode_mode;
  return fuse_scene(j, report);
}

// One scene per GPU at a time: worker d takes the next scene of the list, fuses it on devices[d], repeats.  No data-path
// collective (SURVEY.md §8e): the scenes are independent.
int scn_fuse_many(const char* const* sens_paths, const char* const* out_plys, uint32_t n_scenes, const scn_tsdf_params* params,
                  const int* devices, uint32_t n_devices, const char* decode_mode, scn_fuse_report_t* reports) {
  if (!sens_paths || !params || (!devices && n_devices) || !n_devices) return scn::fail(SCN_ERR_ARG, "null argument");
  std::atomic<uint32_t> next{0}; std::atomic<int> rc{0};
  std::mutex em; std::string first_err;
  auto worker = [&](int dev) {
    for (;;) {
      const uint32_t i = next.fetch_add(1);
      if (i >= n_scenes) break;
      SceneJob j; j.sens_path = sens_paths[i]; j.out_path = out_plys && out_plys[i] ? out_plys[i] : ""; j.params = *params; j.device = dev; j.verbose = false;
      j.decode_mode = decode_mode;
      scn_fuse_report_t r; memset(&r, 0, sizeof(r));
      const int e = fuse_scene(j, &r);
      r.status = e;
      if (reports) reports[i] = r;
      if (e) { std::lock_guard<std::mutex> l(em); if (!rc.load()) { first_err = scn_last_error(); rc.store(e); } }
    }
  };
  std::vector<std::thread> th;
  for (uint32_t d = 1; d < n_devices; ++d) th.emplace_back(worker, devices[d]);
  worker(devices[0]);
  for (auto& t : th) t.join();
  return rc.load() ? scn::fail(rc.load(), "%s", first_err.c_str()) : SCN_OK;
}

int scn_fuse_main(int argc, const char** argv) {
  std::vector<std::string> params, scenes; std::string out_path; int gpus = 0;
  for (int i = 1; i < argc; ++i) {
    const std::string a = argv[i];
    if (a == "--gpus" && i + 1 < argc) { gpus = atoi(argv[++i]); continue; }
    if (a.size() > 5 && a.substr(a.size() - 5) == ".sens") scenes.push_back(a);
    else if (!scenes.empty()) out_path = a;
    else params.push_back(a);
  }
  if (scenes.empty()) {
    printf("Usage: fuse <params.txt> [<params2.txt>] <file.sens> [out.ply]\n       fuse --gpus N <params.txt> ... <a.sens> <b.sens> ...\n");
    return 255;
  }
  scn_tsdf_params p; scn_tsdf_default_params(&p);
  p.max_blocks = 1ull << 22; p.hash_slots = 1ull << 24;      // 16 GiB of voxel blocks unless the parameter file says otherwise (s_hashNumSDFBlocks)
  for (const std::string& f : params) if (scn_tsdf_params_from_file(f.c_str(), &p)) { fprintf(stderr, "%s\n", scn_last_error()); return 1; }
  p.batch_frames = 32;
  const char* mode = getenv("SCN_FUSE_DECODE");
  if (scenes.size() == 1 && gpus <= 1) {
    SceneJob j; j.sens_path = scenes[0]; j.out_path = out_path.empty() ? default_out(scenes[0]) : out_path; j.params = p; j.device = 0; j.verbose = true; j.decode_mode = mode;
    scn_fuse_report_t r;
    if (fuse_scene(j, &r)) { fprintf(stderr, "%s\n", scn_last_error()); return 1; }
    if (getenv("SCN_TIMING"))
      fprintf(stderr, "[timing] fuse %.3f s (waiting for the decoders %.3f s; depth decode %.3f s, colour decode %.3f s on their threads), marching cubes %.3f s, PLY %.3f s, total %.3f s, %.2f GB of HBM in use\n",
              r.fuse_s, r.decode_wait_s, r.depth_decode_s, r.color_decode_s, r.mc_s, r.ply_s, r.total_s, r.device_bytes_in_use / 1e9);
    return 0;
  }
  int ndev = scn_device_count();
  if (ndev <= 0) { fprintf(stderr, "%s\n", scn_last_error()); return 1; }
  if (gpus <= 0 || gpus > ndev) gpus = ndev;
  gpus = std::min<int>(gpus, (int)scenes.size());
  std::vector<const char*> sp, op; std::vector<std::string> outs; std::vector<int> devs;
  for (const std::string& s : scenes) outs.push_back(default_out(s));
  for (size_t i = 0; i < scenes.size(); ++i) { sp.push_back(scenes[i].c_str()); op.push_back(outs[i].c_str()); }
  for (int d = 0; d < gpus; ++d) devs.push_back(d);
  std::vector<scn_fuse_report_t> reps(scenes.size());
  const double t0 = now_s();
  const int rc = scn_fuse_many(sp.data(), op.data(), (uint32_t)scenes.size(), &p, devs.data(), (uint32_t)devs.size(), mode, reps.data());
  const double dt = now_s() - t0;
  uint64_t frames = 0;
  for (size_t i = 0; i < scenes.size(); ++i) {
    const scn_fuse_report_t& r = reps[i];
    printf("%s: GPU %d, %llu frames in %.3f s = %.1f frames/s incl. decode, mesh %llu vertices / %llu faces%s\n", scenes[i].c_str(), r.device,
           (unsigned long long)r.frames_integrated, r.fuse_s, r.frames_integrated / std::max(r.fuse_s, 1e-9), (unsigned long long)r.mesh_vertices,
           (unsigned long long)r.mesh_faces, r.status ? "  FAILED" : "");
    frames += r.frames_integrated;
  }
  printf("%zu scenes on %d GPUs: %llu frames in %.3f s wall = %.1f frames/s aggregate (file -> TSDF -> mesh)\n", scenes.size(), gpus, (unsigned long long)frames, dt, frames / std::max(dt, 1e-9));
  if (rc) { fprintf(stderr, "%s\n", scn_last_error()); return 1; }
  return 0;
}

}  // extern "C"
