/* scannet_b200 — C ABI of the B200-native ScanNet hot path.
 *
 * The reference toolkit exposes NO plugin / operator / FFI interface (SURVEY.md §8b): its
 * seams are three command-line tools and two C++ function/class seams.  Each entry point
 * below names the reference interface it stands in for (paths relative to /root/reference).
 *
 * Conventions: plain C, opaque handles, int status (0 = ok, <0 = error; text via
 * scn_last_error(), thread-local), caller-owned output buffers unless stated, no
 * exceptions cross the boundary, one CUDA stream per handle, handles are not thread-safe.
 * Every compute entry point runs on the GPU; there is no CPU fallback — without a usable
 * CUDA device the call fails with SCN_ERR_CUDA.
 */
#ifndef SCANNET_B200_H
#define SCANNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCN_OK              0
#define SCN_ERR_ARG        -1   /* bad argument */
#define SCN_ERR_CUDA       -2   /* CUDA runtime / no device */
#define SCN_ERR_IO         -3   /* file could not be opened / read / written */
#define SCN_ERR_FORMAT     -4   /* malformed .sens / .ply / .obj / parameter file */
#define SCN_ERR_CAPACITY   -5   /* hash table or block heap exhausted */
#define SCN_ERR_UNSUPPORTED -6  /* e.g. TYPE_OCCI_USHORT depth (needs uplink codec, sensorData.h:711-722) */

const char* scn_last_error(void);
int  scn_version(void);
/* Number of CUDA devices visible (<0 on error). */
int  scn_device_count(void);
/* Creates the CUDA context now (≈0.3 s in a cold process); safe to call from a helper thread while input files are read. */
int  scn_cuda_warmup(void);
/* The batch decoders (scn_inflate_batch_device, scn_jpeg_decode_batch_device) keep their pinned upload slices and device scratch
 * buffers, and scn_fuse_* its frame arrays and its last volume, in per-device pools for the life of the process; this frees the
 * idle ones of the current device. */
int  scn_release_cached_staging(void);
/* Pinned host memory for frame staging (cudaHostAlloc); integrate calls detect it and skip the bounce copy. */
void* scn_host_alloc(size_t bytes);
void  scn_host_free(void* p);
void  scn_free(void* p);                      /* frees buffers this library malloc'ed for the caller */
/* device memory / stream helpers for callers without a CUDA runtime of their own (buffers for scn_sens_decode_depth_device and
 * scn_tsdf_integrate_device); the copies return when the transfer has completed */
void* scn_device_alloc(size_t bytes);
void  scn_device_free(void* p);
int   scn_set_device(int device);                     /* cudaSetDevice for the calling thread (multi-GPU drivers) */
int   scn_device_mem_info(size_t* used_bytes, size_t* total_bytes);
int   scn_stream_create(void** stream_out);          /* non-blocking cudaStream_t */
void  scn_stream_destroy(void* stream);
int   scn_memcpy_h2d(void* d_dst, const void* src, size_t bytes, void* stream);
int   scn_memcpy_d2h(void* dst, const void* d_src, size_t bytes, void* stream);

/* ===================================================================== Segmentator ====
 * Replaces: std::vector<int> segment(const std::string&, float, int)   Segmentator/segmentator.cpp:123
 *           universe* segment_graph(int, int, edge*, float)            Segmentator/segmentator.cpp:71
 *           main / writeToJSON                                         Segmentator/segmentator.cpp:253-288
 */

/* Mesh loading with the same acceptance rules as the reference loader (tinyply path
 * segmentator.cpp:130-140: vertex x,y,z must be 4-byte floats, face list property
 * "vertex_indices" or "vertex_index" with 4-byte indices, triangles only; OBJ path :141-172:
 * original vertices, first shape only).  Buffers are malloc'ed; release with scn_free. */
int scn_mesh_load(const char* path, float** xyz, uint64_t* n_verts, uint32_t** tri, uint64_t* n_faces);

/* flags for scn_segment_mesh */
#define SCN_SEG_DEFAULT        0
#define SCN_SEG_DEVICE_UNIONFIND 1  /* run the Kruskal pass (S5) with the speculative-window device kernel instead of the host loop (default: host; see DESIGN.md §5 for the measured comparison) */
/* test hook (scn_segment_graph only): override introsort's depth limit 2*floor(log2 n) to reach the heap-sort fallback */
#define SCN_SEG_TEST_DEPTH(d)  (((d) & 0xFF) << 8)

/* segment() over raw arrays: seg_out[v] = root vertex id of v's segment, bit-identical to the
 * reference compiled with libstdc++ (incl. std::sort's unstable tie order). */
int scn_segment_mesh(const float* xyz, uint64_t n_verts, const uint32_t* tri, uint64_t n_faces,
                     float k_thresh, int32_t seg_min_verts, int32_t* seg_out, int flags);

/* Intermediates for parity tests: 12-byte {float w; int32 a; int32 b} records, 3 per face,
 * before and after the sort (either pointer may be NULL). */
int scn_segment_mesh_debug(const float* xyz, uint64_t n_verts, const uint32_t* tri, uint64_t n_faces,
                           float k_thresh, int32_t seg_min_verts, int32_t* seg_out, int flags,
                           void* edges_presort, void* edges_sorted, float* vertex_normals,
                           int32_t* roots_after_kruskal);

/* segment_graph(): sorts `edges` (12-byte records) in place exactly like the reference and
 * returns find(v) / size(find(v)) for every vertex after the thresholded Kruskal pass. */
int scn_segment_graph(int32_t n_verts, int64_t n_edges, void* edges, float c,
                      int32_t* roots_out, int32_t* sizes_out, int flags);

/* writeToJSON(): one-line JSON, same byte layout as segmentator.cpp:253-266. */
int scn_write_segs_json(const char* path, const char* scene_id, float k_thresh, int32_t seg_min_verts,
                        const int32_t* seg_indices, uint64_t n);

/* The CLI in library form: `segmentator input.ply [kThresh] [segMinVerts]` (same stdout
 * lines, same output file name <base>.<%f kThresh>.segs.json). Returns the process exit code. */
int scn_segmentator_main(int argc, const char** argv);

/* per-stage timings of the last scn_segment_* call on this thread, milliseconds:
 * [0] H2D, [1] normals, [2] weights, [3] sort, [4] kruskal, [5] small-merge, [6] labels+D2H, [7] total */
int scn_segment_last_timings(float* ms8);
/* rounds taken by the device union-find replay (SCN_SEG_DEVICE_UNIONFIND) in the last scn_segment_mesh call on this thread; 0 = host loop */
uint64_t scn_segment_last_uf_rounds(void);

/* ===================================================================== SensReader =====
 * Replaces: ml::SensorData                                  SensReader/c++/src/sensorData.h:285-1936
 *   ctor/loadFromFile :855,:1250   decompressDepthAlloc :939-946   decompressColorAlloc :929-936
 *   saveToFile :1101-1109          saveToImages :1380-1466         operator<< :1941-1955
 */
typedef struct scn_sens scn_sens;

typedef struct {
  uint32_t version;                 /* 4 */
  uint32_t color_width, color_height, depth_width, depth_height;
  int32_t  color_compression;       /* -1 unknown, 0 raw, 1 png, 2 jpeg   (sensorData.h:346-351) */
  int32_t  depth_compression;       /* -1 unknown, 0 raw u16, 1 zlib u16, 2 occi u16 (:352-357) */
  float    depth_shift;
  uint64_t n_frames, n_imu_frames;
  float    color_intrinsic[16], color_extrinsic[16], depth_intrinsic[16], depth_extrinsic[16];
  char     sensor_name[256];
} scn_sens_info_t;

int  scn_sens_open(const char* path, scn_sens** out);
void scn_sens_close(scn_sens* s);
int  scn_sens_info(const scn_sens* s, scn_sens_info_t* info);
/* camera-to-world (row-major 4x4; all -inf = invalid) + timestamps + compressed sizes */
int  scn_sens_frame_meta(const scn_sens* s, uint64_t frame, float cam2world[16], uint64_t* ts_color,
                         uint64_t* ts_depth, uint64_t* color_bytes, uint64_t* depth_bytes);
/* decoded depth, depth_width*depth_height uint16 (0 = invalid), caller-owned buffer */
int  scn_sens_frame_depth_u16(const scn_sens* s, uint64_t frame, uint16_t* out);
/* decoded colour, color_width*color_height*3 RGB8, caller-owned buffer */
int  scn_sens_frame_color_rgb8(const scn_sens* s, uint64_t frame, uint8_t* out);
/* raw compressed payloads (pointers into the handle; valid until scn_sens_close) */
int  scn_sens_frame_payload(const scn_sens* s, uint64_t frame, const uint8_t** color, const uint8_t** depth);

/* ---- colour decode on the device (R4: sensorData.h:609-616 -> stb_image) ----------------------------------------------
 * n baseline JPEG payloads (host pointers), every one width x height, decoded by the GPU (csrc/jpeg_gpu.cu), byte-identical
 * to scn_sens_frame_color_rgb8 / the reference's stb_image path.
 *   d_lut == NULL : d_out (device) receives n frames of width*height RGB8;
 *   d_lut != NULL : device array of out_px ints = colour pixel index per output pixel (-1 = none -> black); d_out receives n
 *                   frames of out_px RGB8 (colour registered to the depth image, what scn_tsdf_integrate_device consumes).
 * Streams the device path does not handle (progressive, multi-scan, exotic sampling) or flags as corrupt go through the host
 * decoder and are uploaded: same bytes, same errors.  *n_on_device (optional) = frames decoded by the GPU.  `stream` =
 * cudaStream_t (0 = default); returns after the work has completed. */
int scn_jpeg_decode_batch_device(const uint8_t* const* src, const uint64_t* src_bytes, uint32_t n, uint32_t width, uint32_t height,
                                 const int32_t* d_lut, uint32_t out_px, void* d_out, void* stream, uint32_t* n_on_device);
/* timings of the calling thread's last scn_jpeg_decode_batch_device: host parse + pack + upload issue (s), entropy+IDCT kernel (ms), colour kernel (ms) */
int scn_jpeg_last_timings(double* host_s, double* entropy_ms, double* color_ms);
/* colour frames [first, first+n) of an open stream into device memory (JPEG on the GPU; raw / PNG via the host decoder) */
int scn_sens_decode_color_device(const scn_sens* s, uint64_t first, uint32_t n, const int32_t* d_lut, uint32_t out_px, void* d_out,
                                 void* stream, uint32_t* n_on_device);
/* Read-ahead decoder: the counterpart of SensorData::RGBDFrameCacheRead (sensorData.h:1717-1835), which the reconstruction
 * binaries pull frames from.  Background threads (the reference has one; n_threads <= 0 picks min(8, cores)) decode depth and
 * colour of up to cache_size frames ahead of the consumer, in stream order.  scn_sens_cache_next copies the next frame into the
 * caller's buffers (either may be NULL) and returns 1, returns 0 after the last frame, negative on a decode error of that
 * frame.  The scn_sens handle must outlive the cache and must not be modified while it exists. */
typedef struct scn_sens_cache scn_sens_cache;
int  scn_sens_cache_create(const scn_sens* s, uint32_t cache_size, int n_threads, scn_sens_cache** out);
int  scn_sens_cache_next(scn_sens_cache* c, uint16_t* depth_out, uint8_t* color_rgb8_out, uint64_t* ts_depth, uint64_t* ts_color);
void scn_sens_cache_destroy(scn_sens_cache* c);
/* replace a frame's pose (as `recons` writes optimised trajectories back, zParametersScanNet.txt:5) */
int  scn_sens_set_pose(scn_sens* s, uint64_t frame, const float cam2world[16]);
int  scn_sens_save(const scn_sens* s, const char* path);
/* saveToImages(): _info.txt, frame-%06d.color.{jpg,png}, .depth.pgm (P5, 16-bit BE), .pose.txt */
int  scn_sens_save_to_images(const scn_sens* s, const char* out_dir);
/* operator<< text (header summary) into a caller buffer; returns needed length */
int64_t scn_sens_describe(const scn_sens* s, char* buf, uint64_t cap);

/* Writer (initDefault + addFrame + saveToFile pattern, sensorData.h:888-929; Converter/main.cpp:32-41) */
int  scn_sens_create(uint32_t color_w, uint32_t color_h, uint32_t depth_w, uint32_t depth_h,
                     const float color_intrinsic[16], const float depth_intrinsic[16],
                     int32_t color_compression, int32_t depth_compression, float depth_shift,
                     const char* sensor_name, scn_sens** out);
/* colour: raw RGB8 (color_compression 0) or an already-encoded JPEG/PNG payload of color_bytes bytes */
int  scn_sens_add_frame(scn_sens* s, const uint8_t* color, uint64_t color_bytes, const uint16_t* depth,
                        const float cam2world[16], uint64_t ts_color, uint64_t ts_depth);
/* The CLI in library form: `sens <file.sens> [outDir=./out/]` (SensReader/c++/src/main.cpp:28-97). */
int  scn_sens_main(int argc, const char** argv);

/* ===================================================================== TSDF fusion =====
 * Replaces: the external FriedLiver.exe / DepthSensing.exe stage
 *   Server/scan_processor.py:27-35,123-138   (`<exe> <params.txt> <params2.txt> <file.sens>` -> .ply)
 * whose source is NOT in the reference tree.  Numerical spec: DESIGN.md "TSDF spec v1".
 */
typedef struct scn_tsdf scn_tsdf;

typedef struct {
  float    voxel_size;                /* s_SDFVoxelSize               (BASELINE.json: 0.004)           */
  float    trunc_base;                /* s_SDFTruncation                                                */
  float    trunc_scale;               /* s_SDFTruncationScale (m per m of depth)                        */
  float    depth_min, depth_max;      /* s_sensorDepthMin/Max         zParametersScanNet.txt:34-35      */
  float    max_integration_distance;  /* s_SDFMaxIntegrationDistance  :51                               */
  uint32_t weight_sample;             /* s_SDFIntegrationWeightSample :52                               */
  uint32_t weight_max;                /* s_SDFIntegrationWeightMax    :53 (clamped to 255: u8 weight)   */
  uint32_t width, height;             /* integration resolution (BASELINE.json: 640x480)                */
  float    depth_shift;               /* .sens header depthShift (1000)                                 */
  uint64_t hash_slots;                /* open-addressing slots (rounded up to a power of two)           */
  uint64_t max_blocks;                /* 8^3 voxel blocks in the heap (4 KiB each)  s_hashNumSDFBlocks  */
  uint32_t batch_frames;              /* frames fused per block residency, 1..32                        */
  uint32_t flags;                     /* SCN_TSDF_* */
  uint32_t depth_filter;              /* s_depthFilter: bilateral pre-filter of the depth map (zParametersBundlingScanNet.txt:74) */
  float    depth_sigma_d;             /* s_depthSigmaD  (:72) pixels                                    */
  float    depth_sigma_r;             /* s_depthSigmaR  (:73) metres                                    */
} scn_tsdf_params;

#define SCN_TSDF_NO_STATS   1u        /* skip the per-launch counters (N_u, N_b) */
#define SCN_TSDF_KERNEL_TMA    4u     /* always use the cp.async.bulk (TMA) staged integrate kernel (default: only for batches of <= 2 frames) */
#define SCN_TSDF_KERNEL_COLUMN 8u     /* always use the register-resident column kernel */

typedef struct {
  uint64_t frames_integrated, frames_skipped;   /* skipped = invalid (-inf) pose */
  uint64_t blocks_allocated;                    /* live blocks in the heap */
  uint64_t voxels_updated;                      /* Σ_frames N_u */
  uint64_t blocks_visited;                      /* Σ_frames N_b */
  uint64_t algorithmic_bytes;                   /* Σ_frames 2WH + 3WH[colour] + 16 N_u + 16 N_b (SURVEY.md §8d) */
  uint64_t kernel_launches;                     /* kernels this handle launched so far */
  uint32_t error_flags;                         /* bit0 heap full, bit1 table full */
} scn_tsdf_stats_t;

void scn_tsdf_default_params(scn_tsdf_params* p);
/* `key = value;` parameter files as consumed by the external binaries (Server/tools/recons/zParameters*.txt);
 * unknown keys are ignored, known ones override *p. */
int  scn_tsdf_params_from_file(const char* path, scn_tsdf_params* p);
int  scn_tsdf_create(const scn_tsdf_params* p, int device, scn_tsdf** out);
void scn_tsdf_destroy(scn_tsdf* t);
/* Use an existing CUDA stream (cudaStream_t cast to void*; NULL = legacy default stream). */
int  scn_tsdf_set_stream(scn_tsdf* t, void* cuda_stream);
/* One frame from HOST buffers: depth W*H u16, rgb W*H*3 (nullable; must already be registered to
 * the depth image), cam2world row-major 4x4, K = 4x4 depth intrinsic as in the .sens header.
 * Frames whose pose is invalid (cam2world[0] == -inf) are skipped. Asynchronous. */
int  scn_tsdf_integrate(scn_tsdf* t, const uint16_t* depth, const uint8_t* rgb,
                        const float cam2world[16], const float K[16]);
/* n frames from HOST buffers (contiguous frames; poses n*16); H2D copies are pipelined against the
 * kernels.  Identical results to n calls of scn_tsdf_integrate. */
int  scn_tsdf_integrate_batch(scn_tsdf* t, uint32_t n, const uint16_t* depth, const uint8_t* rgb,
                              const float* cam2world, const float K[16]);
/* n frames whose depth/rgb already live in DEVICE memory (poses stay on the host). */
int  scn_tsdf_integrate_device(scn_tsdf* t, uint32_t n, const uint16_t* d_depth, const uint8_t* d_rgb,
                               const float* cam2world, const float K[16]);
int  scn_tsdf_sync(scn_tsdf* t);
int  scn_tsdf_reset(scn_tsdf* t);
int  scn_tsdf_stats(scn_tsdf* t, scn_tsdf_stats_t* out);
/* Optional per-kernel timing: when enabled, CUDA events are recorded on the handle's stream around the
 * alloc and integrate kernels of every batch; scn_tsdf_kernel_times sums them (ms) since enabling.
 * union_blocks = Σ_launches blocks read+written by the integrate kernel (actual 8 KiB/block traffic). */
int  scn_tsdf_profile(scn_tsdf* t, int enable);
int  scn_tsdf_kernel_times(scn_tsdf* t, double* alloc_ms, double* integrate_ms, uint64_t* n_batches,
                           uint64_t* union_blocks);
/* Copies up to `cap` blocks to the host: block_xyz 3*n int32 block coordinates, voxels n*512
 * records of {float sdf; uint8 r,g,b,weight}, x fastest.  Order is heap order (unspecified). */
int  scn_tsdf_download_blocks(scn_tsdf* t, int32_t* block_xyz, void* voxels, uint64_t cap, uint64_t* n);
/* Marching-cubes surface of the current volume (malloc'ed; scn_free).  rgb may be NULL. */
int  scn_tsdf_extract_mesh(scn_tsdf* t, float** xyz, uint8_t** rgb, uint32_t** tri,
                           uint64_t* n_verts, uint64_t* n_faces);
/* PLY writer in the VCGLIB layout Segmentator reads (Server/config/scan_stages.json:33-37). */
int  scn_mesh_save_ply(const char* path, const float* xyz, const uint8_t* rgb, uint64_t n_verts,
                       const uint32_t* tri, uint64_t n_faces);
/* Depth bilateral filter as BundleFusion applies it before integration (zParametersBundlingScanNet.txt:72-74); the only
 * in-tree statement of the kernel is AnnotationTools/Filter2dAnnotations/filter.cu:210-247 (bilateralFilterFloatMapDevice),
 * whose arithmetic (float domain weight, double range weight, -inf = invalid) is reproduced.  depth: w*h uint16 (host);
 * out_metres: w*h float (host), -inf where invalid.  Used inside scn_tsdf_integrate* when params.depth_filter != 0. */
int  scn_depth_bilateral_filter(const uint16_t* depth, uint32_t w, uint32_t h, float depth_shift, float sigma_d, float sigma_r,
                                float* out_metres);
/* ------------------------------------------------------------------------------------------------------------------
 * segs.json consumers (SURVEY.md §8f-4): what the annotation tools do with Segmentator's output.
 * ------------------------------------------------------------------------------------------------------------------ */
/* Reader with the tolerance of AnnotationTools/common/Segmentation.h:57-88: segIndices entries may be JSON ints, uints,
 * strings of digits, or null (-> 0xFFFFFFFF); params.kThresh / params.segMinVerts default to 0 when absent.
 * *seg_out is malloc'ed (release with scn_free); scene_id may be NULL. */
int  scn_segs_load(const char* path, uint32_t** seg_out, uint64_t* n_out, float* k_thresh, uint32_t* seg_min_verts,
                   char* scene_id, size_t scene_id_cap);
/* Segmentation::m_segIdsToVertIds (Segmentation.h:70-75) and computeSurfaceAreaPerSegment (Segmentation.h:113-147) in one pass
 * on the GPU.  Outputs (malloc'ed, scn_free): seg_ids[nS] ascending; vert_offsets[nS+1] + vert_ids[nV]: the vertices of
 * segment k are vert_ids[vert_offsets[k] .. vert_offsets[k+1]) in ascending order (the reference's push_back order);
 * area[nS]: sum of Trianglef::getArea (mLib core-graphics/triangle.h:23-35) over the faces whose three corners all lie in the
 * segment, accumulated in double in ascending face order (the reference adds floats in unordered_map order, so only a
 * tolerance is meaningful).  xyz/tri/area may be NULL/0 to skip the area. */
int  scn_segs_aggregate(const uint32_t* seg, uint64_t n_verts, const float* xyz, const uint32_t* tri, uint64_t n_faces,
                        uint32_t** seg_ids, uint64_t* n_segs, uint64_t** vert_offsets, uint32_t** vert_ids, float** area);
/* Per-vertex object ids from an aggregation (Visualizer.cpp:284-297): group g lists segment ids
 * group_segs[group_offsets[g] .. group_offsets[g+1]); every vertex of those segments gets object id g+1, later groups
 * overwrite earlier ones, vertices of ungrouped segments get 0. */
int  scn_segs_objects_per_vertex(const uint32_t* seg, uint64_t n_verts, const uint32_t* group_segs, const uint64_t* group_offsets,
                                 uint64_t n_groups, uint32_t* obj_out);
/* mLib MeshData::computeVertexNormals (core-mesh/meshData.h:758-782): unit face normals summed per vertex in face order,
 * then normalised with 1/length — bit-identical to the sequential loop. */
int  scn_mesh_vertex_normals(const float* xyz, uint64_t n_verts, const uint32_t* tri, uint64_t n_faces, float* normals_out);
/* Annotation propagation from the decimated to the hi-res mesh (Visualizer::propagateAnnotations, Visualizer.cpp:308-377):
 * for each destination vertex the 3 nearest LABELLED (obj > 0) source vertices decide its object id — the first of them
 * that is closer than maxThresh = max(0.01 * largest source bbox extent, 0.05) and whose normal is within normal_thresh
 * radians wins; otherwise the nearest one's id if all three are within maxThresh and agree; otherwise 0.
 * The reference searches with an approximate FLANN kd-tree; this is the exact 3-NN (ties by source index). */
int  scn_propagate_labels(const float* src_xyz, const float* src_normals, const uint32_t* src_obj, uint64_t n_src,
                          const float* dst_xyz, const float* dst_normals, uint64_t n_dst, float normal_thresh,
                          uint32_t* dst_obj_out);
/* ------------------------------------------------------------------------------------------------------------------
 * GPU depth decode (SURVEY.md §8f-2): TYPE_ZLIB_USHORT payloads (sensorData.h:703-709) are uploaded compressed and inflated
 * in device memory, one warp per frame.  d_depth_out: device pointer, n * depth_width * depth_height uint16, frame after
 * frame — exactly what scn_tsdf_integrate_device consumes.  `stream` is a cudaStream_t (NULL = default stream); the call
 * returns when the frames are decoded.  Same bytes and the same error cases as scn_sens_frame_depth_u16.
 * ------------------------------------------------------------------------------------------------------------------ */
int  scn_sens_decode_depth_device(const scn_sens* s, uint64_t first_frame, uint32_t n, uint16_t* d_depth_out, void* stream);
/* the same for caller-supplied zlib streams: src[i] / src_bytes[i] on the host, each must inflate to >= frame_bytes */
int  scn_inflate_batch_device(const uint8_t* const* src, const uint64_t* src_bytes, uint32_t n, uint64_t frame_bytes, void* d_out,
                              void* stream);
/* timings of the calling thread's last scn_inflate_batch_device: host packing + upload issue (s), kernel (ms, CUDA events), whether
 * the shared-memory-window kernel ran (else the window lives in HBM), streams in the launch */
int  scn_inflate_last_timings(double* pack_s, double* kernel_ms, int* ring_window, uint32_t* n_streams);
/* host build of the same decoder source (one lane): used by the CPU test-suite; not a product path */
int  scn_inflate_host(const uint8_t* src, size_t n, uint8_t* out, size_t cap, size_t* produced);

/* ------------------------------------------------------------------------------------------------------------------
 * Scene fusion driver: .sens -> hashed TSDF -> (optionally) marching cubes -> <out>.ply — the contract of the reference's
 * external reconstruction stage (Server/scan_processor.py:27-35,123-138), one scene per GPU (Server/process.py:75 runs one
 * scan per GPU at a time; SURVEY.md §8e).  decode_mode: NULL = automatic, "gpu" = compressed payloads decoded in HBM,
 * "host" = host thread pool.
 * ------------------------------------------------------------------------------------------------------------------ */
typedef struct scn_fuse_report {
  int32_t  status;                 /* 0 or the error code of this scene (scn_fuse_many) */
  int32_t  device;
  int32_t  gpu_decode;             /* 1 = payloads were decoded on the GPU */
  uint32_t volume_reused;          /* the pooled volume of the previous scene on this GPU was reset instead of a new one created */
  uint32_t color_frames_on_device; /* JPEG frames the device decoder handled itself (the rest went through the host decoder) */
  uint64_t frames_integrated, frames_skipped, frames_skipped_pose;
  uint64_t blocks_allocated, voxels_updated;
  uint64_t mesh_vertices, mesh_faces;
  uint64_t device_bytes_in_use;    /* cudaMemGetInfo after fusion: volume + decode staging */
  double   fuse_s;                 /* first frame in -> last frame integrated, decode included */
  double   decode_wait_s;          /* of which the integrator waited for the decoders */
  double   depth_decode_s, color_decode_s;   /* busy time of the two decoder threads (overlaps fuse_s); host decode: its one thread in depth_decode_s */
  double   integrate_s;            /* integrator: submit + wait for the GPU, all chunks */
  double   depth_pack_s, depth_kernel_s;     /* of depth_decode_s: host packing + upload issue, inflate kernel (CUDA events) */
  double   color_host_s, color_entropy_s, color_convert_s;   /* of color_decode_s: host parse + pack, Huffman+IDCT kernel, colour kernel */
  double   setup_s;                /* open + parse the file, create the volume */
  double   buffers_s, teardown_s;  /* of fuse_s: allocating the double-buffered frame arrays; joining the decoders and freeing them */
  double   mc_s, ply_s, total_s;   /* marching cubes, PLY write, everything incl. opening the file */
} scn_fuse_report_t;
int  scn_fuse_scene(const char* sens_path, const char* out_ply /* NULL: no mesh */, const scn_tsdf_params* params, int device,
                    const char* decode_mode, scn_fuse_report_t* report);
/* n_scenes scenes over n_devices GPUs, one scene per GPU at a time, no data-path collective; reports[i] per scene */
/* sizeof(scn_fuse_report_t) of the library build, for bindings that mirror the struct (tests/test_abi_cpu.py) */
size_t scn_fuse_report_sizeof(void);
int  scn_fuse_many(const char* const* sens_paths, const char* const* out_plys /* NULL or per-scene NULL: no mesh */, uint32_t n_scenes,
                   const scn_tsdf_params* params, const int* devices, uint32_t n_devices, const char* decode_mode,
                   scn_fuse_report_t* reports);
/* `fuse <params.txt> <file.sens> [out.ply]` — the recons/improve stage contract; `fuse --gpus N <params.txt> a.sens b.sens ...` */
int  scn_fuse_main(int argc, const char** argv);

#ifdef __cplusplus
}
#endif
#endif /* SCANNET_B200_H */
