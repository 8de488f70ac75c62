/*
 * voxcarve.h — C ABI of the B200-native voxel-carving engine (libvoxcarve.so).
 *
 * The reference (alxfox/AR_Voxel_Project) has no FFI layer: its hot path is four free
 * functions on `Model&` called from main.cpp:260-303. This header is the boundary a thin
 * C++ shim with those exact signatures binds to (include/voxcarve_shim.hpp, INTEGRATION.md).
 * Each entry point names the reference interface it replaces (paths under src/).
 *
 * Conventions: plain pointers and sizes only; every function returns an int status
 * (VC_OK = 0); no exceptions cross the boundary; output buffers are caller-allocated;
 * an engine is not thread-safe (the reference is single-threaded, Benchmark.h:59-63); engines on DIFFERENT devices may be driven
 * from different threads, engines on the SAME device share its __constant__ view tables and must be driven from one thread at a
 * time (the library orders their launches: a new owner of the tables waits for the previous owner's kernels);
 * all device memory is owned by the engine unless bound with vc_bind_volumes.
 * There is NO CPU fallback: without a CUDA device every call fails with VC_ERR_CUDA.
 *
 * Device-resident grid layout (replaces Model::voxels alpha + Model::seen, Model.h:100-102):
 *   word[(z*Y + y)*Wx + (x >> 5)], bit (x & 31), Wx = ceil(X/32); 1 = occupied / seen.
 *   Row padding bits (x >= X) are always 0. z is the slowest index, as in Model::flatten
 *   (Model.h:104-106), so a z-slab is one contiguous range and slabs gather in place.
 */
#ifndef VOXCARVE_H
#define VOXCARVE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VC_API_VERSION 3

#if defined(__GNUC__)
#define VC_EXPORT __attribute__((visibility("default")))
#else
#define VC_EXPORT
#endif

typedef struct vc_engine vc_engine; /* opaque */

enum vc_status {
    VC_OK = 0,
    VC_ERR_ARG = 1,      /* bad argument (message in vc_last_error) */
    VC_ERR_CUDA = 2,     /* CUDA runtime error, or no device */
    VC_ERR_STATE = 3,    /* call order: views/masks/images not set, halo planes missing, ... */
    VC_ERR_CAPACITY = 4, /* caller buffer too small */
    VC_ERR_COMM = 5      /* NCCL: library not loadable, or a collective failed */
};

/* Grid = Model(x, y, z, size) (Model.h:108, Model.cpp:9-14) restricted to the z-slab
 * [z_begin, z_end) this engine carves. Single GPU: z_begin = 0, z_end = Z. */
typedef struct vc_grid_desc {
    int32_t X, Y, Z;
    float voxel_size;
    int32_t z_begin, z_end;
    int32_t device; /* CUDA ordinal */
} vc_grid_desc;

/* Arithmetic of the projection (VoxelCarving.cpp:18-21).
 * VC_EXACT reproduces the reference bit for bit: f32 world coords, f64 sequential
 * accumulation of the 3x4.4x1 product rounded once to f32, IEEE f32 divides, round half away.
 * It is built from explicit intrinsics, so nvcc's -fmad setting cannot change it.  VC_EXACT classifies
 * 32x8x8-voxel bricks per view first (conservatively, against a summed-area table of the silhouette)
 * and evaluates only the undecided (brick, view) pairs per voxel, each voxel-view first through an f32 filter with a
 * rigorous error radius and exactly (f64) only where the filter cannot tell the pixel; VC_EXACT_FLAT evaluates every
 * voxel-view exactly until its run is empty.  Both produce the same bits.
 * VC_FAST_F32 is a diagnostic f32/FMA pipeline (not bit-exact; see tests/test_fast_mode.py). */
enum vc_carve_mode { VC_EXACT = 0, VC_FAST_F32 = 1, VC_EXACT_FLAT = 2 };
/* values of the reference's -color flag (main.cpp:30,278-288) */
enum vc_color_mode { VC_COLOR_CLOSEST = 1, VC_COLOR_AVG = 2 };
enum vc_mask_format { VC_MASK_BITS = 0, VC_MASK_BGR8 = 1, VC_MASK_BGR8_RAW = 2 /* distorted: undistorted on the device, needs vc_set_calibration */ };
/* Raw (distorted) input - VC_MASK_BGR8_RAW masks, vc_set_images_raw, vc_append_views with raw masks, vc_undistort_bgr - is
 * undistorted on the device bit for bit as cv2 4.13.0's cv::undistort computes it on x86-64 with its AVX2 code path (DESIGN
 * section 8 f-4).  cv::undistort refuses images with a side of 32767 or more (remap's SHRT_MAX limit), so those calls return
 * VC_ERR_ARG for W or H above VC_RAW_MAX_SIDE and leave the engine as it was. */
#define VC_RAW_MAX_SIDE 32766

typedef struct vc_stats {
    double last_carve_ms;          /* CUDA-event time of the last vc_carve (all its kernels) */
    double last_classify_ms;       /* of which (profiling mode only, else 0): the two brick-classification kernels and, on a fresh carve,
                                      the blind fill in front of them; the rest is the per-voxel kernel, whose first blocks also run
                                      the patch pass */
    uint64_t nominal_voxel_views;  /* X*Y*(z_end-z_begin)*V of the last vc_carve */
    uint64_t executed_voxel_views; /* projections actually evaluated, incl. brick corners (0 unless counting was on) */
    uint64_t brick_corner_views;   /* the part of executed_voxel_views spent on brick classification */
    uint64_t bricks_total;         /* bricks of the slab / bricks that needed per-voxel work in the last VC_EXACT carve (with more
                                      than 256 views: summed over the view groups, so a brick listed in two groups counts twice) */
    uint64_t bricks_listed;
    uint64_t flood_rounds;         /* sweep rounds of the last vc_fast_carve */
    uint64_t carve_launches;       /* kernel launches issued by this engine so far */
    uint64_t l2_persist_bytes;     /* always 0 (reserved: keeps the layout of API version 3) */
    /* per-voxel f32 filter of VC_EXACT (counting runs only): 32-voxel rows evaluated, rows that needed the exact f64
     * re-evaluation, and filter decisions that disagreed with the exact evaluation (every decision is cross-checked
     * in a counting run; anything but 0 is a bug) */
    uint64_t filter_rows;          /* in units of 32 voxel-views (one warp instruction stream) */
    uint64_t filter_slow_rows;
    uint64_t filter_mismatches;
    uint64_t subbrick_corner_views; /* the part of brick_corner_views spent inside vc_carve_bricks (8x8x8 sub-brick level) */
    uint64_t volumes_compressible;  /* 1: the engine-owned volumes live in compressible device memory (cuMemCreate, generic compression),
                                       0: plain cudaMalloc memory (not granted by the GPU, or VOXCARVE_COMPRESSIBLE=0 in the environment) */
} vc_stats;

/* ---- lifetime -------------------------------------------------------------------- */
VC_EXPORT int vc_create(const vc_grid_desc* grid, vc_engine** out);
VC_EXPORT void vc_destroy(vc_engine* e);
/* message of the last failed call on `e`; with e == NULL, of the last failed vc_create */
VC_EXPORT const char* vc_last_error(const vc_engine* e);
VC_EXPORT int vc_api_version(void);
/* run all work of this engine on a caller stream (cudaStream_t as void*; NULL = engine's own).  The engine's own stream does
 * not synchronise with other streams, so a caller whose producers (e.g. of device masks) run on its own stream passes that
 * stream here: device pointers are read in the order of the engine's stream only. */
VC_EXPORT int vc_set_stream(vc_engine* e, void* cuda_stream);
VC_EXPORT int vc_synchronize(vc_engine* e);
/* Profiling mode (off by default).  Off: a whole-range VC_EXACT carve is launched as ONE cached CUDA graph (counter reset + the
 * blind fill of a fresh carve on a branch of its own + the two classification kernels + the per-voxel kernel; re-captured
 * whenever grid, slab, views, buffers or stream arguments change; VOXCARVE_NO_GRAPH=1 in the environment disables it) and
 * vc_stats.last_classify_ms stays 0.  On: plain launches in stream order with an event between classification and per-voxel
 * kernel, so that vc_stats splits the carve time and ncu sees every launch.
 * The only other environment switch, read once per process: VOXCARVE_COMPRESSIBLE=0 (engine-owned volumes in plain cudaMalloc
 * memory, what a GPU that refuses compressible memory gets anyway). */
VC_EXPORT int vc_set_profiling(vc_engine* e, int32_t on);

/* ---- inputs ---------------------------------------------------------------------- */
/* Per-view camera data, cached once per dataset (replaces the per-call
 * estimatePoseFromImage + pose.inv() of VoxelCarving.cpp:25-30, ColorReconstruction.h:17-21):
 *   P[v] = intr(CV_32F) * pose(3x4)  — first product of VoxelCarving.cpp:19, 12 f32 row-major
 *   M[v] = pose(3x4) world->camera   — only its translation column is used (ColorReconstruction.h:21);
 *          may be NULL if no colour pass is run. All pointers are HOST memory.
 * Accepted: V in [1,256]; W, H in [1,2^20]; pitch*(H+1) < 2^31 with pitch = 32*(ceil(W/32)+1) (32-bit row offsets of a
 * view's summed-area table); V*H*ceil(W/32) < 2^31 mask words.  Anything else returns VC_ERR_ARG and changes nothing: the
 * engine keeps its previous views, masks, tables and images.  An accepted call replaces every view, also on an engine that
 * vc_append_views had grown past 256: afterwards it holds exactly these V views. */
VC_EXPORT int vc_set_views(vc_engine* e, int32_t V, int32_t W, int32_t H, const float* P, const float* M);
/* More views than one vc_set_views takes: appends views [V, V+n) of the engine's W x H geometry, up to VC_MAX_TOTAL_VIEWS in all.
 * P (and M) hold n*12 floats as in vc_set_views; M must be given if and only if the engine's views have M.  masks: the n new
 * masks in a format of vc_set_masks (VC_MASK_BITS also takes a DEVICE pointer; VC_MASK_BGR8_RAW needs vc_set_calibration, and
 * then images_bgr are raw too, undistorted on the device).  images_bgr: the n new 8UC3 images, required if and only if the
 * engine holds images (vc_set_images / vc_set_images_raw).  Only the new views' summed-area tables are built; the masks, tables
 * and images of the earlier views, the volumes, colour records, mesh and .off text stay as they were, so a capture can grow
 * while the volumes stay on the device: carve just the new frames onto them with vc_carve(e, mode, V_old, -1, 0).
 * Views are processed in groups of 256 consecutive views (one constant-memory batch each); carving is order-independent, and
 * vc_color makes one pass over all views in order, so every result equals that of one engine holding all views at once.
 * VC_ERR_STATE before vc_set_views + vc_set_masks, or for raw masks without calibration; VC_ERR_ARG for n < 1, V+n above
 * VC_MAX_TOTAL_VIEWS, (V+n)*H*ceil(W/32) >= 2^31 mask words, or an M / images_bgr that does not match the engine.  Every check
 * runs and every buffer is allocated before any state changes: a refused call (a failed allocation too) leaves the engine as
 * it was. */
#define VC_MAX_TOTAL_VIEWS 4096
VC_EXPORT int vc_append_views(vc_engine* e, int32_t n, const float* P, const float* M, const void* masks, int32_t mask_format,
                              const uint8_t* images_bgr);
/* vc_set_masks, vc_set_images, vc_set_images_raw, vc_download_masks and vc_download_images take or deliver all V views of the
 * engine, also more than 256 after vc_append_views. */
/* Undistorted silhouette masks (VoxelCarving.cpp:36). VC_MASK_BITS: uint32[V][H][ceil(W/32)],
 * bit x&31 of word x>>5, 1 = background (pixel == (0,0,0), VoxelCarving.cpp:50).
 * VC_MASK_BGR8: the 8UC3 images themselves, uint8[V][H][W][3]; packed on the device. HOST memory (VC_MASK_BITS also takes a
 * DEVICE pointer: silhouettes that a segmentation stage left on the GPU; it is read in the order of the engine's stream only, so
 * their producer runs on that stream, vc_set_stream, or the caller synchronises first).  Builds the summed-area tables of the silhouettes that
 * VC_EXACT's classifier reads (a copy + two kernels, C4: 0.16 ms). */
VC_EXPORT int vc_set_masks(vc_engine* e, const void* masks, int32_t format);
/* Undistorted colour images 8UC3 BGR (ColorReconstruction.h:23), uint8[V][H][W][3], HOST memory. */
VC_EXPORT int vc_set_images(vc_engine* e, const uint8_t* images_bgr);
/* Camera calibration for the on-device cv::undistort (VoxelCarving.cpp:36; ColorReconstruction.h:23): K = 3x3 camera matrix,
 * dist = (k1 k2 p1 p2 [k3 [k4 k5 k6]]) as read from cameracalibration.yml (aruco_samples_utility.hpp:9-16), n_dist in {4,5,8}. */
VC_EXPORT int vc_set_calibration(vc_engine* e, const double K[9], const double* dist, int32_t n_dist);
/* Raw (distorted) colour images as cv::imread delivers them; undistorted on the device, bit-exact with cv::undistort. */
VC_EXPORT int vc_set_images_raw(vc_engine* e, const uint8_t* images_bgr);
/* what the device holds after vc_set_masks / vc_set_images*: bit masks uint32[V][H][ceil(W/32)], images uint8[V][H][W][3] */
VC_EXPORT int vc_download_masks(vc_engine* e, uint32_t* bits);
VC_EXPORT int vc_download_images(vc_engine* e, uint8_t* images_bgr);
/* cv::undistort of n 8UC3 images, HOST in / HOST out, on `device` (utility; the engine paths above keep the data on the GPU). */
VC_EXPORT int vc_undistort_bgr(int32_t device, int32_t n, int32_t W, int32_t H, const uint8_t* src, const double K[9], const double* dist,
                               int32_t n_dist, uint8_t* dst);

/* ---- the hot path ---------------------------------------------------------------- */
/* Model constructor state (Model.cpp:9-14): every voxel occupied, none seen. */
VC_EXPORT int vc_reset(vc_engine* e);
/* carve() (VoxelCarving.h:19, VoxelCarving.cpp:60-72) over views [view_begin, view_end) on this
 * engine's slab; accumulates into the current volumes (call vc_reset first for a fresh Model).
 * view_end < 0 means V. count_executed != 0 also fills vc_stats.executed_voxel_views (slower). */
VC_EXPORT int vc_carve(vc_engine* e, int32_t mode, int32_t view_begin, int32_t view_end, int32_t count_executed);
/* carve() over all views followed by the download of both volumes into HOST buffers, as the shim needs them.  The slab is
 * carved in z-chunks and every finished chunk is copied on a second stream while the next one is carving, so the
 * PCIe transfer overlaps the kernels.  Same result as vc_carve + vc_download_occupied + vc_download_seen. */
VC_EXPORT int vc_carve_download(vc_engine* e, int32_t mode, uint32_t* occupied, uint32_t* seen, uint64_t n_words);
/* (the overlap needs PAGE-LOCKED buffers - cudaHostAlloc / cudaHostRegister: a copy into pageable memory blocks the host, so with
 * pageable buffers the call degrades to the plain carve + two downloads.) */
/* carve() over all views of a FRESH Model (vc_reset pending) + download of the result in SPARSE form: after a fresh carve
 * most 32x8x8-voxel bricks are uniform (C4: 96 %) and one flag byte says everything about them; only the bricks the engine
 * evaluated voxel by voxel need their words.  C4: 0.5 MB + 10 MB over PCIe instead of 268 MB.  With more than 256 views no
 * single classification pass describes the result: the flags are then derived from the carved volumes, and the listed bricks
 * are exactly those that are neither carved whole nor untouched with uniform seen (in no particular order).
 *   brick_flags[b], b = bx + nbx*(by + nby*bz) (vc_sparse_dims; brick = voxels [32bx, 32bx+32) x [8by, 8by+8) x slab planes
 *     [8bz, 8bz+8)): bit 0 (1) = every voxel carved (occupied 0, seen 1), bit 1 (2) = every voxel seen, bit 3 (8) = listed;
 *     a brick that is neither carved nor listed is untouched (occupied 1), one that is not listed has seen = bit 1.
 *   listed[i] = index of the i-th listed brick; words[128 i + r] = its occupied word of row r = 8*plane + y (0 outside the
 *     grid), words[128 i + 64 + r] = its seen word.  n_listed > listed_capacity -> VC_ERR_CAPACITY (the volumes stay on the
 *     device and vc_download_* still works).  include/voxcarve_host.hpp expands this into a Model or into plain words. */
VC_EXPORT int vc_sparse_dims(const vc_engine* e, uint32_t* nbx, uint32_t* nby, uint32_t* nbz);
VC_EXPORT int vc_carve_download_sparse(vc_engine* e, uint8_t* brick_flags, uint64_t flags_capacity, uint32_t* listed, uint32_t* words,
                                       uint64_t listed_capacity, uint64_t* n_listed);
/* fastCarve() (VoxelCarving.h:31, VoxelCarving.cpp:74-167): starts from the Model constructor state (it resets the
 * volumes itself) and needs the whole grid on this engine.  Refused (a slab engine, no views or masks, an unknown mode), it
 * leaves the volumes as they were. */
VC_EXPORT int vc_fast_carve(vc_engine* e, int32_t mode);
/* reconstructClosestColor / reconstructAvgColor (ColorReconstruction.h:131,142): colours every
 * surface voxel (alpha != 0 && !isInner, ColorReconstruction.h:46) of this slab. */
VC_EXPORT int vc_color(vc_engine* e, int32_t color_mode);
/* Occlusion-aware colouring: like vc_color, but a surface voxel takes its colour only from the views that see it.  The records
 * are those of vc_color (same voxels, same order, rgbn.w = min(#observations, 255), MODEL_COLOR with n = 0 when no view
 * observes the voxel), so vc_surface_count, vc_download_colors and apply_colors of vc_dense_from_volumes / vc_mesh_from_volumes
 * take them unchanged.  For each surface voxel (x, y, z) and view v:
 *   1. Sample points: the voxel and its 8 corners (x +- 1/2, y +- 1/2, z +- 1/2), world w = (fl(y' s), fl(x' s), fl(-z' s), 1)
 *      in f32, each projected with the carve's arithmetic (f64 sequential accumulation rounded once to f32 p0, p1, p2; IEEE f32
 *      u = p0/p2, v = p1/p2).  The centre's projection is exactly vc_color's.
 *   2. The pair is eligible iff all 9 points have p2 > 0 and finite u, v (the reference has no depth test and point-reflects
 *      voxels behind the camera; here they neither occlude nor observe).
 *   3. key = min of the 9 p2; rectangle = [round(min u), round(max u)] x [round(min v), round(max v)], round half away from
 *      zero, clipped to the image.
 *   4. Depth buffer per view: zbuf = min(zbuf, key) over every eligible pair and every pixel of its rectangle, from +inf
 *      (order-independent, so the result is deterministic).
 *   5. An eligible pair observes iff its centre pixel (vc_color's pixel) is inside the image and
 *      key <= fl(zbuf[pixel] + tau), tau = fl(tolerance * voxel_size).  A voxel never hides itself (tolerance >= 0).
 *   6. The colour bodies of vc_color run unchanged over the observations only, in view order.
 * tolerance is in voxel sizes.  For P = K [R|t] with K's last row (0, 0, 1), p2 is the camera-space depth in world units, so
 * the tolerance is a depth distance; 2 (the default of the bindings) lets neighbouring voxels of one surface, whose depths
 * differ by up to sqrt(3) voxels, see past each other's corners.  tolerance = +inf keeps every eligible pair whose centre is
 * in the image: where every camera has the whole grid in front of it, that is exactly vc_color.
 * Memory: the records, V * ceil(n_surface / 32) words of observation bits, and depth buffers (4 W H bytes per view) for as many
 * views at a time as 256 MiB holds (at least one); the results do not depend on that chunking.  Works with any number of views.
 * VC_ERR_ARG: mode not 1 or 2, tolerance NaN or negative.  VC_ERR_STATE: a slab engine (whole grid only: occluders in other
 * slabs are unknown), no views or images, or views without M.  These refusals leave the previous records as they were. */
VC_EXPORT int vc_color_visible(vc_engine* e, int32_t color_mode, float tolerance);
/* Cube-index classification of marchingCubes() (MarchingCubes.cpp:12-18, MarchingCubes.h:479-488,
 * :537-552) for the cells whose lower z-plane lies in this slab (plus z = -1 on the first slab). */
VC_EXPORT int vc_mc_classify(vc_engine* e);

/* ---- multi-GPU plumbing ---------------------------------------------------------- */
/* Balanced contiguous z-slabs for n_parts GPUs.  Runs only the two brick-classification passes of VC_EXACT over this
 * engine's z-range (needs views + masks, allocates no volumes; with more than 256 views once per group of 256, the costs summed),
 * takes the per-voxel work left per layer of 8 planes (undecided views x voxels of the listed bricks) and returns n_parts+1 boundaries (interior ones multiples of 8 planes
 * from z_begin) with z_bounds[0] = z_begin, z_bounds[n_parts] = z_end.
 * Deterministic: every rank computes the same split from the same inputs. */
VC_EXPORT int vc_plan_slabs(vc_engine* e, int32_t n_parts, int32_t* z_bounds);
/* Re-range an engine to the slab [z_begin, z_end) of the same grid, keeping views, masks and SAT (plan on the whole grid,
 * then narrow). The volumes are reset. */
VC_EXPORT int vc_set_slab(vc_engine* e, int32_t z_begin, int32_t z_end);
/* Use caller-owned device buffers holding the WHOLE grid (Z*Y*Wx words each); the engine
 * carves its slab in place at word offset z_begin*Y*Wx, so an all-gather of the slabs is in
 * place, and colour / MC passes read neighbour planes from the gathered buffer. */
VC_EXPORT int vc_bind_volumes(vc_engine* e, void* d_occupied_full, void* d_seen_full);
/* device pointers of this engine's slab (first word of plane z_begin) */
VC_EXPORT int vc_device_volumes(vc_engine* e, void** d_occupied_slab, void** d_seen_slab);
/* declare that planes outside the slab held in a bound full volume are valid (after the gather) */
VC_EXPORT int vc_set_gathered(vc_engine* e, int32_t gathered);

/* Whole-grid buffers owned by the engine (instead of caller-owned ones, vc_bind_volumes): what vc_gather fills. Resets the state. */
VC_EXPORT int vc_alloc_full_volumes(vc_engine* e);

/* One-plane halos.  The consumers of a slab read ONE neighbour plane of `occupied` on each side: isInner of the colour pass
 * (Model.h:126-132) planes z_begin - 1 and z_end, the cube index (MarchingCubes.h:537-552) plane z_end.  A plane is Y*Wx words
 * (vc_halo_words).  Planes outside the grid are empty by definition (Model::get, Model.h:119-124) and never exchanged.
 * Imported halos stay valid until this engine carves / resets / uploads again (its neighbours then carve again too).
 *   vc_export_halo: device pointer of the slab's own first (which = 0) or last (which = 1) plane.
 *   vc_import_halo: copy a plane (device pointer on any GPU of this process; the copy runs on this engine's stream, the
 *                   caller orders it after the producer) into plane z_begin - 1 (which = 0) or z_end (which = 1); NULL drops it.
 *   vc_exchange_halos_peer: all engines of ONE process (any devices, any order; their slabs must tile a z-range): every
 *                   engine receives its neighbours' boundary planes, ordered after the producers' streams by events.
 *   vc_exchange_halos: the same across processes / threads over NCCL send/recv, rank r holding the slab below rank r + 1. */
VC_EXPORT int vc_halo_words(const vc_engine* e, uint64_t* n_words);
VC_EXPORT int vc_export_halo(vc_engine* e, int32_t which, void** d_plane);
VC_EXPORT int vc_import_halo(vc_engine* e, int32_t which, const void* d_plane);
VC_EXPORT int vc_exchange_halos_peer(vc_engine** engines, int32_t n);
/* vc_gather (below) for the engines of ONE process without NCCL: every engine pulls the other slabs into its whole-grid buffers
 * with peer copies over NVLink on its own stream (peer access is enabled on the way), ordered after the producers by events.
 * what: 1 = occupied, 2 = seen, 3 = both.  The slabs must tile [0, Z). */
VC_EXPORT int vc_gather_peer(vc_engine** engines, int32_t n, int32_t what);

/* NCCL communicator of the engines that share one grid, one rank per GPU, slabs in rank order along z (SURVEY §8b "gather()").
 * libnccl.so.2 is loaded at run time, the first time one of these is called (a copy the process already carries - a
 * Python framework may bundle its own - is shared); VC_ERR_COMM if it cannot be.  Rank 0 makes the 128-byte id with vc_comm_unique_id and hands it to
 * the other ranks by any means (MPI, a file, a socket); vc_comm_init blocks until all `world` ranks have called it.
 *   vc_exchange_halos: see above.  One grouped send/recv pair per neighbour on the engine's stream; returns without waiting.
 *   vc_gather: assemble the whole grid in place in the whole-grid buffers (vc_alloc_full_volumes / vc_bind_volumes) of
 *     every rank.  what: 1 = occupied, 2 = seen, 3 = both; z_bounds = the world + 1 slab boundaries (vc_plan_slabs).  Equal
 *     slabs: one in-place ncclAllGather per volume; balanced (ragged) slabs: one group of sends / receives per volume.
 *     Marks the grid gathered (vc_set_gathered) when `occupied` was included.  Only a consumer that needs every voxel - the
 *     host Model, fastCarve's flood - needs this; colour and cube-index passes need the halos only.
 *   vc_comm_allreduce_u64: element-wise sum of n host counters over the ranks (cube-index histograms, voxel counts). */
VC_EXPORT int vc_comm_unique_id(void* unique_id_128);
VC_EXPORT int vc_comm_init(vc_engine* e, int32_t rank, int32_t world, const void* unique_id_128);
VC_EXPORT int vc_comm_destroy(vc_engine* e);
VC_EXPORT int vc_comm_info(const vc_engine* e, int32_t* rank, int32_t* world, int32_t* nccl_version);
VC_EXPORT int vc_exchange_halos(vc_engine* e);
VC_EXPORT int vc_gather(vc_engine* e, int32_t what, const int32_t* z_bounds);
VC_EXPORT int vc_comm_allreduce_u64(vc_engine* e, uint64_t* values, int32_t n);
/* The WHOLE grid (Z*Y*Wx words) out of the whole-grid buffers into HOST memory: which = 0 occupied (must have been gathered),
 * 1 seen (gathered by the caller's choice of vc_gather's `what`).  What the shim fills a host Model from after vc_gather. */
VC_EXPORT int vc_download_full(vc_engine* e, int32_t which, uint32_t* words, uint64_t n_words);

/* ---- outputs (HOST buffers, caller-allocated) ------------------------------------ */
VC_EXPORT int vc_slab_words(const vc_engine* e, uint64_t* n_words); /* (z_end-z_begin)*Y*Wx */
/* Load this slab's volumes from HOST words: how the shim hands an existing Model (alpha != 0 and
 * Model::seen, e.g. after applyClosure, main.cpp:297-303) to vc_color / vc_mc_classify. Padding
 * bits are cleared. */
/* A later vc_carve accumulates onto this state exactly like the reference: a voxel that arrives carved but unseen is still
 * marked seen by every view that has it inside the image (VoxelCarving.cpp:45-54). */
VC_EXPORT int vc_upload_volumes(vc_engine* e, const uint32_t* occupied, const uint32_t* seen, uint64_t n_words);
VC_EXPORT int vc_download_occupied(vc_engine* e, uint32_t* words, uint64_t n_words);
VC_EXPORT int vc_download_seen(vc_engine* e, uint32_t* words, uint64_t n_words);
VC_EXPORT int vc_count_occupied(vc_engine* e, uint64_t* n_occupied, uint64_t* n_seen);
/* result of vc_color: one record per surface voxel in ascending flatten order
 * (idx = x + X*(y + Y*z), Model.h:104-106); rgbn = r, g, b, min(#observations, 255);
 * voxels with 0 observations keep MODEL_COLOR (ColorReconstruction.cpp:29-31, Model.h:90). */
VC_EXPORT int vc_surface_count(vc_engine* e, uint64_t* n);
VC_EXPORT int vc_download_colors(vc_engine* e, uint64_t* idx, uint8_t* rgbn, uint64_t capacity);
/* result of vc_mc_classify: histogram of cube indices, #cells with edgeTable[idx] != 0,
 * #triangles (sum of triTable row lengths / 3) */
VC_EXPORT int vc_download_mc(vc_engine* e, uint64_t hist256[256], uint64_t* n_active, uint64_t* n_triangles);
VC_EXPORT int vc_get_stats(vc_engine* e, vc_stats* out);

/* ---- "next" rows: dense RGBA Model on the device, applyClosure, marchingCubes triangles (whole grid only) ---- */
/* Load the reference Model's voxels (its RGBA float vector, X*Y*Z*4 floats, index = Model::flatten, Model.h:100-106). */
VC_EXPORT int vc_dense_upload(vc_engine* e, const float* rgba);
/* Build the Model's voxels from the device volumes: occupied -> MODEL_COLOR, carved -> 0 (Model.h:90, VoxelCarving.cpp:52);
 * apply_colors != 0: the records of the last vc_color (ColorReconstruction.cpp:41,66); handle_unseen != 0:
 * Model::handleUnseen (Model.cpp:36-47). */
VC_EXPORT int vc_dense_from_volumes(vc_engine* e, int32_t apply_colors, int32_t handle_unseen);
/* model.set(x, y, z, (0,0,0,0)) for every voxel the device volumes hold as carved (VoxelCarving.cpp:52), on the dense Model
 * already on the device (vc_dense_upload): the Model after carve() when it held other state before (-intermediateMesh,
 * VoxelCarving.cpp:65-68, takes a mesh of it after every view). */
VC_EXPORT int vc_dense_apply_carved(vc_engine* e);
/* applyClosure(model, kernelSize) (Postprocessing3d.h:10): returns VC_ERR_ARG for an even kernel size (reference: -1). */
VC_EXPORT int vc_dense_closure(vc_engine* e, int32_t kernel_size);
VC_EXPORT int vc_dense_download(vc_engine* e, float* rgba);
/* marchingCubes(model, ..., threshold) geometry (MarchingCubes.h:596, MarchingCubes.cpp:8-19): triangles in the reference's
 * emission order, 3 unshared vertices each (voxel-index coordinates, before WriteMesh's scale/translation) + face colour. */
VC_EXPORT int vc_mc_mesh(vc_engine* e, float threshold, uint64_t* n_triangles);
VC_EXPORT int vc_download_mesh(vc_engine* e, float* verts /* T*9 */, uint32_t* rgb /* T*3 */, uint64_t capacity_triangles);

/* ---- the mesh straight from the bit volumes (main.cpp:291-303 without the dense Model) ---- */
/* marchingCubes of the Model that vc_dense_from_volumes(apply_colors, handle_unseen) [+ vc_dense_closure(closure_k)] would build,
 * computed from the bit volumes and the colour records without the dense Model: the same triangles, vertices and colours in the
 * same order as that chain + vc_mc_mesh(threshold), left in the mesh buffers for vc_download_mesh.  closure_k = 0: no closure;
 * otherwise odd, at most VC_MESH_MAX_CLOSURE (else VC_ERR_ARG).  Every alpha of such a Model is 0 or 1, so the geometry is marching
 * cubes on occupied | ~seen (handle_unseen) dilated by the closure box, and every vertex sits on a voxel; a threshold outside
 * (0, 1] gives no triangles.  Memory: one extra bit volume (closure only), a row table of the colour records (4 (Y*Z+1) bytes),
 * 4 (X+1)(Y+1) bytes of column counts and the mesh; the dense Model is not allocated or touched.
 * VC_ERR_STATE: a slab engine (whole grid only), or apply_colors without a vc_color of the current volumes.
 * VC_ERR_CAPACITY: 2^32 triangles or more.  A refused call leaves the previous mesh as it was. */
#define VC_MESH_MAX_CLOSURE 15
VC_EXPORT int vc_mesh_from_volumes(vc_engine* e, int32_t apply_colors, int32_t handle_unseen, int32_t closure_k, float threshold,
                                   uint64_t* n_triangles);

/* ---- the .off file of the mesh, formatted on the device (SimpleMesh::WriteMesh, MarchingCubes.h:59-87) ---- */
/* The complete text of the file WriteMesh writes for the mesh the last vc_mc_mesh / vc_mesh_from_volumes left on the device:
 * "OFF\n", "3T T 0\n", 3T vertex lines "a b c\n" with a = fl(fl(x * scale) + tx) (no FMA, x86 NaN rules: a NaN operand keeps
 * its sign, 0 * inf and inf - inf give -nan), then T face lines "3 3i 3i+1 3i+2 r g b\n" (rgb printed with %u).  Numbers are
 * printed as a C++ ostream prints a float by default: printf("%g") of the float, 6 significant digits rounded correctly
 * (ties to even) from the exact binary value, "C" locale; denormals, -0, inf, -inf, nan and -nan included.  scale multiplies
 * the voxel-index coordinates of the mesh: the reference's scaleFactor = scale * voxel size (MarchingCubes.cpp:23).
 * The text stays in a grow-only device buffer (n_bytes = its size, at most 39 bytes per vertex line and 71 per face line)
 * until the next call; vc_download_mesh_off copies any byte range of it into HOST memory, so a caller can write the file
 * in chunks.  Refusals leave the previous text as it was: VC_ERR_STATE without a mesh; VC_ERR_CAPACITY above
 * VC_TEXT_MAX_LINES lines (4T lines: T > 2^29 triangles).  vc_download_mesh_off: VC_ERR_STATE when no text was formatted or
 * the mesh has changed since; VC_ERR_ARG for a range that ends past the text. */
#define VC_TEXT_MAX_LINES (1ull << 31) /* what one scan of u32 line lengths takes */
VC_EXPORT int vc_mesh_format_off(vc_engine* e, float scale, float tx, float ty, float tz, uint64_t* n_bytes);
VC_EXPORT int vc_download_mesh_off(vc_engine* e, uint64_t offset, void* dst, uint64_t n_bytes);
/* Utility (HOST in / HOST out, on `device`): one line "%g\n" per value, with the device code of vc_mesh_format_off and no
 * arithmetic on the values.  *n_bytes = the text's size; VC_ERR_CAPACITY (nothing written) when it exceeds `capacity`;
 * at most VC_TEXT_MAX_LINES values. */
VC_EXPORT int vc_format_g(int32_t device, uint64_t n, const float* values, char* text, uint64_t capacity, uint64_t* n_bytes);

/* ---- measurement helper (bench.py roofline denominators) ------------------------- */
/* Register-resident FFMA and DFMA loops on `device`: measured CUDA-core peaks in TFLOP/s
 * (2 flops per FMA), timed with CUDA events, best of 5. Not part of the carve path. */
VC_EXPORT int vc_measure_peaks(int32_t device, double* ffma_tflops, double* dfma_tflops);
/* GPU self-test of the kernel's arithmetic shortcuts over n pseudo-random inputs:
 * which = 0 shared-reciprocal f32 divide vs IEEE div.rn; which = 1 pixel index vs (int)roundf + inside();
 * which = 2 packed f32 pairs (fma / add / mul .rn.f32x2, both halves) vs the scalar IEEE operations.
 * Returns the number of disagreements and of cases compared. */
VC_EXPORT int vc_selftest(int32_t device, int32_t which, uint64_t n, uint64_t seed, uint64_t* mismatches, uint64_t* checked);
/* Probes of the exact carve's two approximations, for tests (HOST in / HOST out, on the engine's stream, synchronised).  They run
 * the compiled code of the carve on records of the caller's choice, with the engine's views (any index in [0, V), including
 * views past 256), masks, summed-area tables, filter constants, voxel size, W, H and slab.
 * vc_probe_boxes: boxes[n][7] = (view, x0, y0, z0, x1, y1, z1), inclusive voxel ranges, global z -> out[n][5] = (code, px0, px1,
 *   py0, py1): the brick classifier's answer (0 undecided, 1 every voxel outside the image, 2 every voxel inside on foreground,
 *   3 inside on background, 4 inside but not decided by the table) and the pixel rectangle it counted in the table (codes 2-4;
 *   zeros otherwise).
 * vc_probe_voxels: voxels[n][4] = (view, x, y, z), global z -> out[n][11] = (decided, inside, px, py) of the per-voxel f32 filter,
 *   (inside, px, py) of the exact evaluation, and the bit patterns of the view's Cu, Cv and the engine's hDu, hDv.  Pixels are
 *   meaningful where inside (and, for the filter, decided).
 * VC_ERR_ARG: a null buffer, more than VC_PROBE_MAX records, a view outside [0, V), a range outside the grid or the slab, or
 * x1 < x0 (y, z alike).  VC_ERR_STATE: no views or no masks.  Nothing is launched on a refused call. */
#define VC_PROBE_MAX (1ull << 26)
VC_EXPORT int vc_probe_boxes(vc_engine* e, uint64_t n, const int32_t* boxes, int32_t* out);
VC_EXPORT int vc_probe_voxels(vc_engine* e, uint64_t n, const int32_t* voxels, int32_t* out);

#ifdef __cplusplus
}
#endif
#endif /* VOXCARVE_H */
