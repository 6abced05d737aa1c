/* dogeray_b200 -- C ABI of the B200-native path tracer that replaces the hot path of
 * PhilipPragerUrbina/DOGERAY's raygpu/kernel.cu (".rts in -> path-traced image out").
 *
 * The reference has no plugin/FFI interface; its de-facto boundary is
 *     cudaError_t CudaStarter(int3* outputr, bvh* nbvhtree, singleobject* allobjects,
 *                             cudaTextureObject_t* texarray, int divisor)
 * (raygpu/kernel.cu:138, :2562-2669) plus the file-scope settings it reads
 * (kernel.cu:29-30, 119-132) and the start-up sequence of main() (kernel.cu:2055-2103:
 * getnum -> read -> readtextures -> build_bvh).  Each entry point below says which of
 * those it replaces.
 *
 * Conventions: plain C types only; every function returns DRB_OK (0) or a negative
 * drb_status and never throws; drb_last_error() holds the message of the last failure
 * on the calling thread.  A drb_scene lives on ONE CUDA device and is not thread-safe
 * (one call at a time per handle).  There is no CPU fallback: without a usable CUDA
 * device every device entry point fails with DRB_ERR_CUDA.
 */
#ifndef DOGERAY_B200_H
#define DOGERAY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRB_ABI_VERSION 2

typedef enum drb_status {
    DRB_OK = 0,
    DRB_ERR_ARG = -1,       /* bad argument */
    DRB_ERR_IO = -2,        /* file cannot be opened / short read / short write */
    DRB_ERR_PARSE = -3,     /* malformed .rts or .ppm content */
    DRB_ERR_CUDA = -4,      /* CUDA runtime error, or no device */
    DRB_ERR_NOMEM = -5,
    DRB_ERR_UNSUPPORTED = -6
} drb_status;

/* ---- the settings line of a .rts file ------------------------------------------------
 * "*,camx,camy,camz,aperture,lookx,looky,lookz,focus,fov,maxdepth,spp,bgintensity,backtex,W,H"
 * (writer plugin/rtsexport.py:207, reader kernel.cu:1223-1299).  Defaults are the
 * file-scope initialisers kernel.cu:29-30, 119-132.  These are also the 13 floats
 * CudaStarter packs into settings[] (kernel.cu:2581). */
typedef struct drb_settings {
    float cam[3];           /* campos            default 0,0,2 */
    float aperture;         /* aperturee         default 0.01  */
    float look[3];          /* look              default 0,0,0 */
    float focus;            /* focus_diste       default 3     */
    int32_t fov;            /* fovv, degrees, vertical; default 45 */
    int32_t max_depth;      /* max_depthh        default 50    */
    int32_t spp;            /* samples_per_pixell default 1    */
    float bg_intensity;     /* backgroundintensity default 1   */
    int32_t backtex;        /* index into the scene's texture table, -1 = sky gradient */
    int32_t width;          /* SCREEN_WIDTH      default 1280  */
    int32_t height;         /* SCREEN_HEIGHT     default 720   */
} drb_settings;

/* ---- one object line of a .rts file ---------------------------------------------------
 * Column meaning: SURVEY.md App. A.2; reader kernel.cu:1316-1503; the in-memory layout the
 * reference parses into is `singleobject` (kernel.cu:48-74).  This struct is the
 * file-format view (what a loader or a scene writer exchanges), not the device layout. */
typedef struct drb_object {
    float pos[3];           /* col 0-2   triangle v0 / sphere centre */
    int32_t type;           /* col 3     0 sphere, 2 triangle */
    float col[3];           /* col 4-6 */
    float add_y;            /* col 7     roughness, or IOR for glass (addional.y) */
    float add_x;            /* col 8     != 0 -> normalised diffuse lobe (addional.x) */
    float dim[3];           /* col 9-11  triangle v1 / sphere radius in [0] */
    int32_t mat;            /* col 12    0 diffuse, 2 mirror, 3 metal, 4 glass, 5 glossy, other emissive */
    float rot[3];           /* col 13-15 triangle v2 */
    float norm[3];          /* col 16-18 face normal, sentinel z == -20 */
    float n1[3], n2[3], n3[3]; /* col 19-27 vertex normals, sentinel z == -20 */
    float t1[2], t2[2], t3[2]; /* col 28-33 UVs, defaults (0,1) (0,0) (1,0) */
    int32_t smooth;         /* col 34 */
    int32_t checker;        /* col 35    `tex` flag: procedural checker */
    int32_t texnum;         /* col 36    colour texture index or -1 */
    int32_t rtexnum;        /* col 37    roughness texture index or -1 */
    int32_t ncols;          /* how many columns the line had (0 for objects made in memory) */
} drb_object;

/* ---- host-side scene description: replaces getnum + read + getppmpaths (kernel.cu:1113-1530,
 * 1979-2018).  Pure host code, no CUDA. ------------------------------------------------- */
typedef struct drb_host_scene drb_host_scene;

/* Parse `rts_path`.  Textures are looked up by name among the files of `tex_dir` whose name
 * contains "ppm"/"PPM" (NULL -> current working directory, as the reference does), visited in
 * sorted order; the lower-cased path must contain the (unmodified) query, kernel.cu:1172-1183. */
int drb_host_scene_load(const char* rts_path, const char* tex_dir, drb_host_scene** out);
/* drb_host_scene_load through a binary cache (SURVEY.md 8(f)1).  The cache file (`cache_path`, NULL ->
 * rts_path + ".drbcache") holds the parsed objects and settings keyed by a 64-bit hash of the scene text, its
 * length, the scanned texture list (texture ids are indices into it) and the ABI version; on any mismatch or
 * damage the text is parsed and the cache rewritten (atomically; failing to write it is not an error).  A hit
 * returns exactly what drb_host_scene_load returns.  *cache_hit (may be NULL) says which happened. */
int drb_host_scene_load_cached(const char* rts_path, const char* tex_dir, const char* cache_path,
                               drb_host_scene** out, int* cache_hit);
/* the content hash the cache is keyed by (chunked multiply-fold, not cryptographic) */
uint64_t drb_hash_bytes(const void* data, size_t len);
/* Same from a memory buffer holding .rts text. */
int drb_host_scene_parse(const char* text, size_t len, const char* tex_dir, drb_host_scene** out);
/* Build one from arrays (synthetic scenes).  `tex_paths` may be NULL when ntex == 0. */
int drb_host_scene_create(const drb_settings* settings, const drb_object* objects, int64_t nobjects,
                          const char* const* tex_paths, int ntex, drb_host_scene** out);
void drb_host_scene_free(drb_host_scene* hs);
int64_t drb_host_scene_num_objects(const drb_host_scene* hs);
const drb_object* drb_host_scene_objects(const drb_host_scene* hs);
int drb_host_scene_settings(const drb_host_scene* hs, drb_settings* out);
int drb_host_scene_num_textures(const drb_host_scene* hs);
const char* drb_host_scene_texture_path(const drb_host_scene* hs, int i);
/* objects that become primitives of the tree (type 0 / 2 with enough columns); counted on first call, then remembered */
int64_t drb_host_scene_num_renderable(const drb_host_scene* hs);
/* lines skipped while parsing (unsupported type, junk line); see drb_last_error() for the first */
int64_t drb_host_scene_num_skipped(const drb_host_scene* hs);
/* Write a scene in the exporter's format (plugin/rtsexport.py:207, 312-314). */
int drb_rts_write(const char* path, const drb_settings* settings, const drb_object* objects, int64_t nobjects,
                  const char* const* tex_names, int ntex, const char* backtex_name);
void drb_settings_default(drb_settings* out);

/* ---- device scene: replaces readtextures + build_bvh + the per-frame upload inside
 * CudaStarter (kernel.cu:1915-1976, 1864-1909, 2604-2629).  Uploads once, builds the LBVH on the
 * GPU, keeps everything resident. ----------------------------------------------------- */
typedef struct drb_scene drb_scene;

int drb_scene_create(const drb_host_scene* hs, int device, drb_scene** out);
/* Same with build flags.  DRB_BUILD_LBVH_ONLY keeps the Karras hierarchy as the traversal tree (fastest
 * build); by default the hierarchy is rebuilt over the same Morton order by SAH-guided agglomerative
 * clustering, which traverses ~1.4x faster. */
#define DRB_BUILD_LBVH_ONLY 1u
/* DRB_BUILD_KEEP_DEBUG keeps the integer outputs of the build (keys, order, both binary hierarchies: ~100 B per
 * primitive) resident for drb_scene_lbvh / drb_scene_tree; without it they are scratch and those getters fail. */
#define DRB_BUILD_KEEP_DEBUG 2u
int drb_scene_create_ex(const drb_host_scene* hs, int device, uint32_t build_flags, drb_scene** out);
/* Same, with the object lines ALREADY in device memory: `objects_dev` points at drb_host_scene_num_objects(hs) records
 * of drb_object on `device`, in file order (e.g. each rank uploaded 1/N of them and one all-gather over NVLink
 * completed the array -- the per-frame upload of CudaStarter, kernel.cu:2604-2629, paid once per node instead of once per
 * GPU).  `stream` (a cudaStream_t, may be NULL) is the stream the array was produced on: the build waits for it.  `hs`
 * supplies settings, textures and counts; the array is only read during the call. */
int drb_scene_create_from_device(const drb_host_scene* hs, int device, uint32_t build_flags, const void* objects_dev, void* stream,
                                 drb_scene** out);
/* The same scene on `ndevices` devices (out[k] on devices[k]; a device may be listed more than once).  The object lines
 * cross PCIe ONCE in total: device k uploads lines [k*chunk, (k+1)*chunk), the devices then pull each other's shares over
 * NVLink (peer copies), and every device builds its own tree.  On failure nothing is left allocated. */
int drb_scene_create_multi(const drb_host_scene* hs, const int* devices, int ndevices, uint32_t build_flags, drb_scene** out);
/* convenience: drb_host_scene_load + drb_scene_create */
int drb_scene_load(const char* rts_path, const char* tex_dir, int device, drb_scene** out);
void drb_scene_free(drb_scene* s);
int drb_scene_settings(const drb_scene* s, drb_settings* out);
int64_t drb_scene_num_prims(const drb_scene* s);       /* primitives in the tree */
int64_t drb_scene_num_objects(const drb_scene* s);     /* object lines (ids index these) */

typedef struct drb_build_info {
    int64_t nprims, nnodes;
    float bounds_min[3], bounds_max[3];
    float upload_ms, build_ms;
    int32_t max_depth;          /* height of the traversal tree */
    int32_t rebuild_iterations; /* clustering rounds of the SAH-guided rebuild (0 with DRB_BUILD_LBVH_ONLY) */
    int64_t nwide;              /* four-wide traversal nodes */
    int32_t wide_levels;        /* height of the four-wide tree */
    int32_t stack_levels;       /* traversal stack entries per lane (exact bound computed by the collapse) */
} drb_build_info;
int drb_scene_build_info(const drb_scene* s, drb_build_info* out);

/* Integer outputs of the GPU LBVH build, for the bit-exact check against a host build (scenes created with
 * DRB_BUILD_KEEP_DEBUG; DRB_ERR_UNSUPPORTED otherwise).  Any pointer may be NULL.  keys: n 64-bit sort keys in sorted order; order: n prim slots in
 * sorted order; parent/left/right: n-1 internal nodes, children >= 0 are internal nodes,
 * children < 0 are leaves encoded as ~sorted_position; node_min/node_max: 3 floats per
 * internal node. */
int drb_scene_lbvh(const drb_scene* s, uint64_t* keys, int32_t* order, int32_t* parent, int32_t* left, int32_t* right,
                   float* node_min, float* node_max);

/* The hierarchy the traversal nodes were emitted from, root = node 0, same child encoding as
 * drb_scene_lbvh; equals the Karras tree with DRB_BUILD_LBVH_ONLY.  For the bit-exact host check (DRB_BUILD_KEEP_DEBUG). */
int drb_scene_tree(const drb_scene* s, int32_t* left, int32_t* right, float* node_min, float* node_max);

/* The four-wide traversal nodes (collapsed from drb_scene_tree's hierarchy): child[4*i + k] is child k of node i
 * (>= 0 wide node, < 0 leaf ~primitive slot, INT32_MIN empty); boxes[12*i + 3*k + a] is min_q | max_q << 16 of
 * that child on axis a (16-bit scene grid).  nwide entries each (drb_build_info.nwide). */
int drb_scene_wide(const drb_scene* s, int32_t* child, uint32_t* boxes);

/* Refit: replace the object lines of a resident scene and update its traversal tree in place.  The tree keeps its
 * topology; only primitives, shading records and node boxes change (no Morton sort, no rebuild, same handle, and the
 * query and render buffers stay).  The traversal cost of the tree grows as the geometry moves away from the arrangement
 * it was built for; rebuild with drb_scene_create_from_device when it has moved far.
 *   objects_dev  `nobjects` records of drb_object in file order, on the scene's device; nobjects must equal
 *                drb_scene_num_objects(s).  Only read during the call.
 *   stream       the stream that produced the array (a cudaStream_t; NULL -> the scene's own).  The refit runs on it,
 *                after that stream's earlier work and after work already enqueued on the scene's own stream.  Work on
 *                other streams that reads the scene must be finished by the caller before the call.
 * Every line that was a renderable triangle or sphere at creation must still be one, of the same kind, no other line may
 * become renderable, and the vertex, centre and radius values of renderable lines must be finite.  Otherwise the call
 * returns DRB_ERR_ARG, drb_last_error() names the first offending line, and the scene is unchanged (every line is checked
 * before anything is written).  Everything else in a line may change: vertices, normals, UVs, colour, roughness,
 * material, texture ids (still indexing the textures uploaded at creation) and flags.  The camera is not part of a refit.
 * One host synchronisation (for the validation result and the new bounds): when the call returns the refit is complete
 * and later work on any stream sees the new scene.  drb_build_info then has the new bounds; every other field keeps its
 * build-time value.  drb_scene_lbvh / drb_scene_tree (DRB_BUILD_KEEP_DEBUG) keep describing the build; drb_scene_wide
 * returns the refitted nodes.  Box for box the result equals quantising the new leaf boxes on the grid of the new
 * bounds and taking the integer union bottom-up over the unchanged links. */
int drb_scene_refit_device(drb_scene* s, const void* objects_dev, int64_t nobjects, void* stream);
/* Same from HOST records: copied into device scratch on the scene's own stream, then as above. */
int drb_scene_refit(drb_scene* s, const drb_object* objects_host, int64_t nobjects);

/* ---- rendering ------------------------------------------------------------------------ */
typedef struct drb_opts {
    uint64_t seed;              /* Philox key */
    uint32_t sample_base;       /* first sample index of this call */
    uint32_t sample_count;      /* samples per pixel to trace in this call; 0 -> settings->spp, unless DRB_FLAG_EXACT_SAMPLES */
    uint32_t batch_paths;       /* paths in flight per wavefront batch (120 B of queues each); 0 -> up to 40 % of device memory */
    uint32_t flags;             /* DRB_FLAG_* */
    void* stream;               /* cudaStream_t to launch on; NULL -> the scene's own (non-blocking) stream.  For the legacy
                                 * default stream pass cudaStreamLegacy, not 0 */
    uint32_t tile_rank;         /* tile sharding: trace only the 8x4-pixel tiles t with t % tile_count == tile_rank;  */
    uint32_t tile_count;        /* pixels of other tiles are left untouched in accum.  0 or 1 -> the whole image      */
} drb_opts;
#define DRB_FLAG_ACCUMULATE 1u  /* add into accum instead of overwriting it */
/* sample_count is taken literally: 0 traces nothing (accum is zeroed, or left alone with DRB_FLAG_ACCUMULATE).  A rank
 * whose share of a sharded frame is empty (spp < ranks, distributed.shard_samples) passes its count with this flag. */
#define DRB_FLAG_EXACT_SAMPLES 2u

typedef struct drb_stats {
    uint64_t paths;             /* camera paths traced */
    uint64_t rays;              /* closest-hit queries (one per hit() call of the reference, kernel.cu:800) */
    float trace_ms;             /* device time of the closest-hit kernel, summed over launches */
    float total_ms;             /* device time of the whole call */
    uint32_t trace_launches;
    uint32_t kernel_launches;
} drb_stats;

void drb_opts_default(drb_opts* out);

/* Replaces the accumulate loop of main() (kernel.cu:2154-2224) and every CudaStarter call in
 * it: traces `sample_count` samples for every pixel and writes the SUM of radiance, row-major,
 * 3 floats per pixel, index (y*W + x)*3, linear, unclamped.  Divide by the sample count for the
 * mean.  accum_dev is a DEVICE pointer (W*H*3 floats).  All work is enqueued on opts->stream (the caller's stream
 * order is respected); the host reads one queue counter per bounce to size the next launches and to stop a batch
 * early, so the call returns after the last batch has been enqueued, not necessarily finished: synchronise the
 * stream (or pass `stats`, which synchronises to fill it) before reading accum_dev. */
int drb_render_device(drb_scene* s, const drb_settings* settings, const drb_opts* opts, float* accum_dev, drb_stats* stats);
/* Same with a HOST accumulation buffer (synchronous; includes the device->host copy). */
int drb_render(drb_scene* s, const drb_settings* settings, const drb_opts* opts, float* accum_host, drb_stats* stats);
/* One frame over several resident scenes -- normally the same scene created on different devices (SURVEY.md
 * 8(b)3 "device list", 8(e); drb_scene_create_multi) -- from one process, one host thread per handle.
 *   default           interleaved tiles: handle k traces the 8x4-pixel tiles t with t % nscenes == k (opts->tile_rank /
 *                     tile_count are overridden).  Pixel sets are disjoint, so the image is bit-identical to drb_render on
 *                     a single handle, with or without DRB_FLAG_ACCUMULATE.
 *   DRB_FLAG_DYNAMIC_TILES   the tiles are cut into 4 x nscenes interleaved shards that the handles claim from a shared
 *                     atomic queue as they become free: a slower or busier GPU takes fewer shards.  Same bits as above.
 *   DRB_FLAG_SHARD_SAMPLES   handle k traces sample range k of nscenes (as the torch.distributed path does); the partial
 *                     sums are added in handle order, so the image equals the one-handle image up to float re-association.
 * The image lives in ONE device buffer on scenes[0]'s device.  Where the devices have peer access (NVLink) the other
 * handles' resolve kernels write their tiles straight into it -- the gather rides on the last kernel of the render, there
 * is no separate exchange step -- and sample shards are summed by one kernel on that device reading the peers' buffers.
 * One host <-> device copy of the image per call in total.  Without peer access the shards are merged through host
 * memory.  opts->stream must be NULL.  `stats`: paths, rays and launches are summed, times are the maximum over handles.
 * (torch.distributed callers use drb_render_device + one NCCL reduce instead, INTEGRATION.md 3.) */
#define DRB_FLAG_DYNAMIC_TILES 4u
#define DRB_FLAG_SHARD_SAMPLES 8u
int drb_render_multi(drb_scene* const* scenes, int nscenes, const drb_settings* settings, const drb_opts* opts,
                     float* accum_host, drb_stats* stats);
/* Per-handle device time (ms) of the last drb_render_multi call on this thread, handle order, up to `n` entries; returns how
 * many handles that call had.  For load-balance measurements. */
int drb_render_multi_times(float* ms, int n);

/* Exact output contract of CudaStarter (kernel.cu:2562-2669, Kernel :998-1093): out[(x*H + y)*3 + c] =
 * trunc(255 * mean radiance) for x < W/divisor/8*8, y < H/divisor/8*8, other entries untouched.
 * `out` is a host buffer of W*H*3 int32. */
int drb_frame_i3(drb_scene* s, const drb_settings* settings, const drb_opts* opts, int divisor, int32_t* out);

/* Closest-hit object ids (index of the object line, -1 = miss) and distances for explicit rays:
 * the same query as hit() (kernel.cu:468-512).  o3/d3: n*3 floats on the host.  Runs drb_trace_device's query on the
 * scene's own stream and returns when the results are in ids / t.  It uses the same query buffers as drb_trace_device and
 * drb_occluded_device (below), so it shares their rule: one call at a time per handle.  A device query enqueued on another
 * stream must have finished before this call. */
int drb_trace_ids(drb_scene* s, const float* o3, const float* d3, int64_t n, int32_t* ids, float* t);

/* ---- ray queries on device arrays ----------------------------------------------------------
 * Both calls take DEVICE arrays on the scene's device, enqueue their work on `stream` (a cudaStream_t; NULL -> the scene's
 * own stream; for the legacy default stream pass cudaStreamLegacy, not 0) and return without synchronising: synchronise
 * the stream before reading the results.  Rays are processed in chunks of DOGERAY_B200_QUERY_CHUNK (default 64 Mi) through
 * query buffers of the scene's own, 40 B per ray of a chunk, kept until drb_scene_free; the render's buffers and results
 * are not touched.  Like drb_render_device: one call at a time per handle, and successive calls on a handle ordered on ONE
 * stream (the buffers are reused by the next call).  n == 0 does nothing; n < 0 or a NULL required pointer -> DRB_ERR_ARG. */

/* Closest hit for n rays, o3_dev / d3_dev n*3 float32: exactly the query of drb_trace_ids / hit() (kernel.cu:468-512),
 * t in (1e-4, 1e4) for triangles, (0, 1e4) for spheres.  ids_dev: object-line index or -1; t_dev (may be NULL): distance,
 * -1 on a miss; uv_dev (may be NULL): n*2 float32, the (u, v) of hit_tri for a triangle hit (hit point =
 * (1-u-v)*v0 + u*v1 + v*v2), (0, 0) for a sphere or a miss. */
int drb_trace_device(drb_scene* s, const float* o3_dev, const float* d3_dev, int64_t n,
                     int32_t* ids_dev, float* t_dev, float* uv_dev, void* stream);
/* Any hit: occluded_dev[i] = 1 if some primitive is accepted by hit()'s test at a distance t < min(tmax_dev[i], 1e4), else 0
 * (so exactly (closest id >= 0) && (closest t < tmax)); tmax <= 0 or NaN gives 0.  tmax_dev == NULL -> 1e4 for every ray.
 * occluded_dev: n bytes (viewable as torch.bool).  Stops at the first accepted primitive. */
int drb_occluded_device(drb_scene* s, const float* o3_dev, const float* d3_dev, const float* tmax_dev, int64_t n,
                        uint8_t* occluded_dev, void* stream);
/* The camera rays of sample `sample` for every pixel, row-major (y*W + x): what Kernel computes at
 * kernel.cu:1067-1076.  o3/d3: W*H*3 floats on the host. */
int drb_primary_rays(drb_scene* s, const drb_settings* settings, const drb_opts* opts, uint32_t sample, float* o3, float* d3);

/* The display transform of main() (kernel.cu:2287): 8-bit = clamp(trunc(255 * sum / nsamples), 0, 255),
 * linear, no gamma.  accum row-major W*H*3 floats (host); rgb8 W*H*3 bytes, row-major, y = 0 at the top. */
int drb_tonemap(const float* accum_host, int width, int height, double nsamples, uint8_t* rgb8);
/* Device variant, asynchronous on `stream`: used after an NCCL reduce on rank 0. */
int drb_tonemap_device(const float* accum_dev, int width, int height, double nsamples, uint8_t* rgb8_dev, void* stream);

/* ---- image files ---------------------------------------------------------------------- */
/* 32-bpp BITMAPV4HEADER BMP exactly as SDL_SaveBMP writes the reference's screenshots
 * (kernel.cu:2505-2513; layout pinned by images/ *.bmp, SURVEY.md App. C.1). */
int drb_write_bmp(const char* path, const uint8_t* rgb8, int width, int height);
int drb_write_ppm(const char* path, const uint8_t* rgb8, int width, int height);
/* P6/P5 -> RGBA8 with alpha 0, rows top-down (what sdkLoadPPM4 hands readtextures, kernel.cu:1926).
 * *rgba is malloc'd; release with drb_free. */
int drb_read_ppm(const char* path, uint8_t** rgba, int* width, int* height);
void drb_free(void* p);

/* ---- misc ------------------------------------------------------------------------------ */
const char* drb_last_error(void);
int drb_abi_version(void);
int drb_device_count(void);
/* Device memory is recycled through a block cache and the stream-ordered pool and is not returned to the driver
 * when scenes are freed; this hands all idle memory of `device` back (call with no render in flight). */
int drb_trim(int device);
/* word `n` of the sampler stream of pixel (x, y), sample `sample` (Philox4x32-10; see DESIGN.md) */
uint32_t drb_philox_word(uint64_t seed, uint32_t x, uint32_t y, uint32_t sample, uint32_t n);

#ifdef __cplusplus
}
#endif
#endif /* DOGERAY_B200_H */
