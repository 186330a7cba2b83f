/*
 * rtrace.h -- C ABI of librtrace_b200.so, the B200 (sm_100a) replacement for the
 * data-parallel hot path of Byron/rust-tracer.
 *
 * Each entry point cites the reference interface it replaces (paths relative to
 * the reference repo).  Conventions: every function returns RT_OK (0) or a
 * negative rt_status; no exception or unwinding crosses this boundary;
 * rt_last_error() returns a thread-local message for the last failure.  The
 * library owns rt_scene and all device memory behind it; the caller owns every
 * output buffer.  Output pointers may be host memory (pageable or pinned) or
 * device memory of the scene's GPU -- the library detects which.  A scene is
 * immutable after creation and bound to the CUDA device that was current when
 * it was created.  There is NO CPU fallback: without a usable CUDA device every
 * compute entry point fails with RT_ERR_CUDA.
 */
#ifndef RTRACE_B200_H
#define RTRACE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID = -1, /* bad argument (the reference would panic: render.rs:265-266, group.rs:59) */
    RT_ERR_CUDA = -2,    /* CUDA runtime / driver failure, or no device              */
    RT_ERR_NOMEM = -3,
    RT_ERR_BUFFER = -4   /* output buffer too small                                  */
} rt_status;

/* Opaque scene: replaces `Scene` (src/rust/render.rs:138-142) and the
 * `SphericalGroup` tree it owns (src/rust/group.rs:16-20,86), flattened once
 * into a pre-order float4 + skip-link array resident in HBM/L2. */
typedef struct rt_scene rt_scene;

/* Camera.  NULL wherever a camera is accepted == the reference's fixed camera:
 * origin `scene.eye`, direction normalize(x-W/2,(H-y)-H/2,W) (render.rs:226-243).
 * A non-NULL camera is an extension (orbit sweep): the camera-space direction is
 * rotated by the basis before normalisation; the identity basis reproduces the
 * reference bit for bit. */
typedef struct rt_camera {
    float eye[3];
    float right[3];
    float up[3];
    float forward[3];
} rt_camera;

/* One ray / one closest-hit record: `Ray` (primitive.rs:9-13), `Hit` (primitive.rs:15-19). */
typedef struct rt_ray { float pos[3]; float dir[3]; } rt_ray;
typedef struct rt_hit { float distance; float normal[3]; } rt_hit; /* distance = +inf on miss */

/* Per-call statistics (optional out-parameter; may be NULL). */
typedef struct rt_stats {
    uint64_t primary_rays; /* W*H*spp^2 of the rendered rows                               */
    uint64_t shadow_rays;  /* samples with a hit and g<0 (render.rs:194-203); 0 unless counted */
    double kernel_ms;      /* device time of the traversal kernel(s), CUDA events           */
    double total_ms;       /* kernel + gather + copy-out, host wall clock                   */
    uint32_t kernel_launches;
    uint32_t gpus;
    uint32_t variant_used; /* RT_VARIANT_* the call actually ran (AUTO resolved; LANE when the arguments leave
                              the candidate-list variants' domain: spp > 8, level > 10, eye inside the root
                              bound, camera basis whose row dot products are more than 1e-6 off orthonormal,
                              scene far from the coordinate origin)                                         */
    uint32_t reserved;
} rt_stats;

/* Kernel variants (rt_set_variant).  All produce identical bytes. */
enum {
    RT_VARIANT_AUTO = 0,  /* the fastest parity-green kernel for the arguments          */
    RT_VARIANT_LANE = 1,  /* one thread per pixel, per-lane skip-pointer traversal      */
    RT_VARIANT_WARP = 2,  /* warp-cooperative traversal (ballot/shuffle)                */
    RT_VARIANT_TILE = 3,  /* tile beam-culling + candidate lists, one fused kernel      */
    RT_VARIANT_PHASED = 4 /* the same algorithm as four homogeneous launches on one stream */
};

/* ---- library ------------------------------------------------------------ */
const char *rt_last_error(void);
const char *rt_version(void);
/* Number of usable CUDA devices (0 if none); never fails. */
int rt_device_count(void);
/* Make `device` the current CUDA device of the calling thread (scenes are created
 * on the current device). */
int rt_set_device(int device);
/* Select the kernel variant used by subsequent render calls on this thread. */
int rt_set_variant(int variant);

/* ---- scene: replaces Scene::default + SphericalGroup::pyramid -------------- */
/* render.rs:145-166 + group.rs:28-66: pyramid(level, origin, radius); the light is
 * normalised exactly as `Vector::normalized` does (vec.rs:93-95).  level must be
 * > 1 (group.rs:59-60 asserts) and <= 12.  Built on the current CUDA device. */
int rt_scene_create(uint32_t level, const float origin[3], float radius,
                    const float light_unnormalised[3], const float eye[3], rt_scene **out);
/* Scene::default(): level 8, origin (0,-1,0), radius 1, light (-1,-3,2), eye (0,0,-4). */
int rt_scene_create_default(rt_scene **out);
/* An arbitrary group tree in pre-order: spheres4 = n x {cx,cy,cz,r}; skip[i] > i+1
 * marks node i as a group bound whose subtree ends before skip[i]; leaves have
 * skip[i] == i+1; node 0 must be a group with skip[0] == n.  Mirrors hand-built
 * groups such as the reference's test fixture (group.rs:118-151). */
int rt_scene_create_from_nodes(uint32_t n, const float *spheres4, const uint32_t *skip,
                               const float light[3], const float eye[3], rt_scene **out);
void rt_scene_destroy(rt_scene *s);
/* group.rs:95-109 `count()` -> (groups, items); pins group.rs:183 (5461, 21845). */
int rt_scene_counts(const rt_scene *s, uint64_t *groups, uint64_t *items);
/* Copy the flattened scene back to the host (n x float4, n x u32); returns the node
 * count through n_out; pointers may be NULL to query the size only. */
int rt_scene_export_nodes(const rt_scene *s, float *spheres4, uint32_t *skip, uint32_t cap, uint32_t *n_out);
/* The same flattening WITHOUT a device (host logic only; used by tools and the CPU
 * test-suite): pyramid(level, origin, radius) -> n x float4 + n x u32.  Pass NULL
 * arrays to query n. */
int rt_flatten_pyramid_host(uint32_t level, const float origin[3], float radius,
                            float *spheres4, uint32_t *skip, uint32_t cap, uint32_t *n_out);
int rt_scene_light(const rt_scene *s, float light[3]);
int rt_scene_eye(const rt_scene *s, float eye[3]);
int rt_scene_device(const rt_scene *s);

/* ---- the hot path ---------------------------------------------------------- */
/* Replaces Renderer::render_region (render.rs:218-255) for the region
 * [l,r) x [b,t) of a width x height image (b = upper image row, as in
 * ImageRegion, render.rs:43-72).  Writes (r-l)*(t-b)*4 bytes RGBA8 row-major from
 * row b (RGBABuffer layout, render.rs:69-71,92-109).  Unlike Renderer::render
 * (render.rs:264-266) sizes need not be multiples of 64.  A region narrower than
 * the image (a bucket) is traced by the per-lane kernel over just its own pixels,
 * so its cost is its area; a full-width region takes the variant AUTO picks. */
int rt_render_region(const rt_scene *s, uint16_t width, uint16_t height, uint16_t spp,
                     uint16_t l, uint16_t b, uint16_t r, uint16_t t,
                     uint8_t *rgba_out, size_t rgba_len);

/* Replaces the bucket loop of Renderer::render (render.rs:268-309) for one GPU's
 * share of a frame: rows row_start, row_start+row_stride, ... (row_count of them),
 * all columns, packed densely with the given pitch in bytes (0 = width*4).
 * `stream` is a cudaStream_t (NULL = default stream); with a device output pointer
 * the call is asynchronous on that stream.  camera may be NULL.  kinds_out
 * (optional, device or host) receives one byte per sample (index ssx*spp+ssy):
 * 0 background, 1 hit facing away from the light, 2 lit, 3 shadowed. */
int rt_render_rows(const rt_scene *s, const rt_camera *camera,
                   uint32_t width, uint32_t height, uint32_t spp,
                   uint32_t row_start, uint32_t row_stride, uint32_t row_count,
                   uint8_t *rgba_out, size_t pitch_bytes, uint8_t *kinds_out,
                   void *stream, rt_stats *stats);

/* rt_render_rows with the rows taken in BLOCKS: local row j is image row
 * row_start + (j / row_block) * row_stride + j % row_block (row_block a power of two,
 * row_stride >= row_block).  Rank r of N renders row_start = r*B, row_stride = N*B: whole tiles
 * stay contiguous in the image, so the tile culls stay as tight as on one GPU.  With
 * absolute_rows != 0, rgba_out is the base of a WHOLE device frame (possibly a peer GPU's, e.g. rank
 * 0's through rt_ipc_open) and row j is stored at rgba_out + image_row * pitch: the kernels' stores are
 * the gather. */
int rt_render_row_blocks(const rt_scene *s, const rt_camera *camera,
                         uint32_t width, uint32_t height, uint32_t spp,
                         uint32_t row_start, uint32_t row_stride, uint32_t row_block, uint32_t row_count,
                         uint8_t *rgba_out, size_t pitch_bytes, int absolute_rows,
                         void *stream, rt_stats *stats);

/* Undersampled preview of a frame (the reference README's "interactive rendering with undersampling",
 * README.md:42-48; no counterpart in render.rs): the image is cut into step x step pixel blocks, the ONE
 * ray of each block's first pixel (its top-left, 1 sample per pixel, exactly Renderer::render_region's value
 * for that pixel at samples_per_pixel = 1) is traced and its colour fills the block.  step = 1 is the
 * plain 1-spp frame; the cost falls with step^2.  rgba_out: host or device buffer of width*height*4 bytes;
 * `stream` as in rt_render_rows (a device output is not synchronised). */
int rt_render_preview(const rt_scene *s, const rt_camera *camera, uint32_t width, uint32_t height, uint32_t step,
                      uint8_t *rgba_out, size_t rgba_len, void *stream);

/* Whole frame to a host or device buffer of width*height*4 bytes on the scene's GPU. */
int rt_render_frame(const rt_scene *s, const rt_camera *camera,
                    uint32_t width, uint32_t height, uint32_t spp,
                    uint8_t *rgba_out, size_t rgba_len, rt_stats *stats);

/* A sweep of n_frames frames (cameras[f], or the reference camera when cameras is
 * NULL), pipelined: two frames render at a time on two streams (the launch tails
 * of frame f are filled by the first launches of frame f+1) while the device-to-host
 * copy of an earlier frame runs on a third.  `cb` is called on the calling thread, in frame order, with a pinned host
 * buffer that stays valid until the callback returns.  The scene's scratch is
 * locked for the whole sweep: the callback must not render with the same scene
 * (other scenes and other threads' calls on this scene simply wait).  This is the end-to-end
 * path of the orbit sweep (BASELINE C5) and what `rtrace --frames` uses. */
typedef void (*rt_frame_callback)(void *user, uint32_t frame, const uint8_t *rgba, size_t len);
int rt_render_sweep(const rt_scene *s, const rt_camera *cameras, uint32_t n_frames,
                    uint32_t width, uint32_t height, uint32_t spp,
                    rt_frame_callback cb, void *user, rt_stats *stats);

/* The same sweep delivering RGB8 frames (width*height*3 bytes): the reference's sink drops the
 * alpha channel anyway (render.rs:389-397), so the frame is packed on the device and a quarter of
 * the PCIe traffic is saved.  The bytes are exactly the body of the P6 file. */
int rt_render_sweep_rgb(const rt_scene *s, const rt_camera *cameras, uint32_t n_frames,
                        uint32_t width, uint32_t height, uint32_t spp,
                        rt_frame_callback cb, void *user, rt_stats *stats);

/* Whole frame on ngpu GPUs of this process: the scene is replicated (scenes[g], all distinct, each on its
 * own device) and GPU g renders blocks of 16 consecutive rows, ngpu blocks apart (whole cull tiles stay
 * together; interleaving balances the uneven flake).  rgba_out in HOST memory (pinned for full speed): every
 * GPU copies its own blocks straight into it over its own PCIe link, all links in parallel -- the host frame
 * is where the bands meet, nothing is gathered on a GPU.  rgba_out in DEVICE memory of scenes[0]'s GPU: the
 * kernels of the other GPUs store their pixels into it through peer memory (NVLink) -- the stores are the
 * gather; without peer access GPU g renders rows g, g+ngpu, ... and a strided peer copy de-interleaves them.
 * Replaces the thread pool + sync_channel of Renderer::render (render.rs:271-307). */
int rt_render_frame_multi(rt_scene *const *scenes, int ngpu, const rt_camera *camera,
                          uint32_t width, uint32_t height, uint32_t spp,
                          uint8_t *rgba_out, size_t rgba_len, rt_stats *stats);

/* ---- float output ----------------------------------------------------------------------------------------------
 * The pixel before quantisation: four f32 per pixel {r, g, b, alpha}, 16 bytes, the sums of the spp*spp samples
 * times 1/(spp*spp) (render.rs:249-250), equal bit for bit to the reference's values.  Blue equals green.
 * Quantising each component with trunc(0.5 + 255 v), saturating to 0..255 (NaN -> 0), gives exactly the RGBA8
 * bytes of rt_render_rows (render.rs:96-103).  Float frames are rendered by the PHASED variant (where AUTO would
 * run TILE or PHASED, and for a forced TILE or PHASED) or by LANE (a forced LANE or WARP, and every argument
 * outside PHASED's domain); stats->variant_used says which.  A device output pointer must be 16-byte aligned and
 * a pitch a multiple of 16, else RT_ERR_INVALID. */
/* rt_render_rows with float output and no kinds_out: rows row_start, row_start+row_stride, ... (row_count of
 * them), pitch in bytes (0 = width*16).  With a device output pointer the call is asynchronous on `stream`
 * (e.g. straight into a torch CUDA tensor on torch's current stream). */
int rt_render_rows_f32(const rt_scene *s, const rt_camera *camera,
                       uint32_t width, uint32_t height, uint32_t spp,
                       uint32_t row_start, uint32_t row_stride, uint32_t row_count,
                       float *rgba_out, size_t pitch_bytes, void *stream, rt_stats *stats);
/* rt_render_frame_multi with float output: rgba_out holds width*height*16 bytes (RT_ERR_BUFFER when rgba_bytes
 * is less), in host memory or in device memory of scenes[0]'s GPU; ngpu == 1 is a single-GPU frame. */
int rt_render_frame_multi_f32(rt_scene *const *scenes, int ngpu, const rt_camera *camera,
                              uint32_t width, uint32_t height, uint32_t spp,
                              float *rgba_out, size_t rgba_bytes, rt_stats *stats);

/* The same sweep with the frames PULLED instead of listed: whenever the pipeline has room for another frame the
 * library calls `next(next_user, &camera, &use_camera)`, which fills the camera (or sets *use_camera = 0 for the
 * reference camera; it is 1 on entry) and returns the frame's id (>= 0; handed back to `cb` as its frame argument)
 * or -1 when there is nothing left.  This is how several GPUs (threads of one process, or
 * one process per GPU sharing a counter in shared memory) draw frames from one queue, so that a GPU with a slower
 * host link simply takes fewer of them -- the reference's pool takes every unit of work the same way
 * (render.rs:273-298).  Frames are delivered in the order they were pulled; rgb != 0 delivers RGB8. */
typedef int (*rt_next_frame_callback)(void *user, rt_camera *camera_out, int *use_camera);
int rt_render_sweep_pull(const rt_scene *s, rt_next_frame_callback next, void *next_user,
                         uint32_t width, uint32_t height, uint32_t spp, int rgb,
                         rt_frame_callback cb, void *user, rt_stats *stats);
/* fetch-and-add on a 64-bit counter in host memory (e.g. a POSIX shared-memory segment the ranks of a job map):
 * the frame queue of a multi-process sweep.  Returns the value before the addition. */
uint64_t rt_atomic_fetch_add_u64(void *addr, uint64_t value);

/* The sweep sharded by FRAME over ngpu GPUs of this process (BASELINE configs[4]; scenes[g] is the replica
 * on its own device, all distinct): every GPU runs its own pipelined sweep (two frames in flight + copy-out, as
 * rt_render_sweep) on its own host thread and takes the next frame of the list whenever its pipeline has room
 * (dynamic: a GPU behind a slower host link takes fewer frames), and `cb` is called on the CALLING thread in
 * frame order 0, 1, 2, ... with a pinned host buffer valid until it returns.  rgb != 0 delivers RGB8 frames as
 * rt_render_sweep_rgb does.  No data-path collective: frames are independent.  Replaces the one pool that takes
 * every unit of work and the bounded channel to the writer (render.rs:271-307).  This is what
 * `rtrace --frames K --gpus N` calls. */
int rt_render_sweep_multi(rt_scene *const *scenes, int ngpu, const rt_camera *cameras, uint32_t n_frames,
                          uint32_t width, uint32_t height, uint32_t spp, int rgb,
                          rt_frame_callback cb, void *user, rt_stats *stats);

/* ---- PNG output, encoded on the GPU ------------------------------------------------------------------------
 * One fixed layout, so there is exactly one file per image (DESIGN.md "PNG output"): 8-bit RGB (alpha dropped, as
 * the P6 sink does), one IDAT chunk per band of 16 rows, every row one byte-aligned fixed-Huffman deflate block of
 * literals and distance-3 matches.  Any PNG decoder reads it. */
/* Worst-case size of rt_encode_png's output for a width x height frame (1..65535 each). */
int rt_png_bound(uint32_t width, uint32_t height, size_t *bytes);
/* PNG file (layout above) of a width x height RGBA8 frame in device memory of the current device
 * (pitch 0 = width*4; alpha is dropped).  png_out: host or device memory.  Waits for `stream` and
 * returns the file length in *len_out; RT_ERR_BUFFER (with *len_out = the needed size) if cap is short;
 * RT_ERR_INVALID for a host rgba pointer or a zero size. */
int rt_encode_png(const uint8_t *rgba, uint32_t width, uint32_t height, size_t pitch_bytes,
                  uint8_t *png_out, size_t cap, size_t *len_out, void *stream);
/* rt_render_sweep_multi delivering each frame as a complete PNG file (len = file size), in frame order,
 * on the calling thread; ngpu == 1 is the single-GPU pipelined sweep.  Each frame is encoded on its GPU behind
 * its render launches and only the file's bytes cross the host link. */
int rt_render_sweep_png(rt_scene *const *scenes, int ngpu, const rt_camera *cameras, uint32_t n_frames,
                        uint32_t width, uint32_t height, uint32_t spp,
                        rt_frame_callback cb, void *user, rt_stats *stats);

/* ---- Animated PNG (APNG) of a sweep, encoded on the GPU ------------------------------------------------------
 * One file per animation, written as one payload per frame (DESIGN.md "Animated PNG"): the file is the payloads of
 * frames 0 .. n_frames-1 back to back.  Each frame's zlib stream is exactly that of its rt_encode_png file.  Frame 0
 * carries the signature, IHDR, acTL (n_frames, loop for ever), its fcTL and its IDAT chunks, so a viewer without
 * APNG support shows frame 0.  Every later frame is an fcTL and the same chunks as fdAT.  The last frame also carries
 * IEND.  Every frame is full size and shows for delay_num / delay_den seconds. */
/* Worst-case payload of one frame of a width x height, n_frames animation (pure arithmetic, no device).
 * RT_ERR_INVALID for a size outside 1..65535, n_frames == 0, or sequence numbers beyond 2^31 - 1. */
int rt_apng_bound(uint32_t width, uint32_t height, uint32_t n_frames, size_t *frame_bytes);
/* Payload of frame `frame` of an n_frames animation from a width x height RGBA8 frame in device memory of the
 * current device.  Errors as rt_encode_png, plus RT_ERR_INVALID when frame >= n_frames.  Uses rt_encode_png's
 * scratch of this (device, stream). */
int rt_encode_apng_frame(const uint8_t *rgba, uint32_t width, uint32_t height, size_t pitch_bytes, uint32_t frame,
                         uint32_t n_frames, uint16_t delay_num, uint16_t delay_den, uint8_t *out, size_t cap,
                         size_t *len_out, void *stream);
/* rt_render_sweep_png delivering each frame's payload instead of a PNG file: the bytes handed to `cb`, concatenated
 * in frame order, are the animation.  Each frame is encoded on the GPU that rendered it. */
int rt_render_sweep_apng(rt_scene *const *scenes, int ngpu, const rt_camera *cameras, uint32_t n_frames,
                         uint32_t width, uint32_t height, uint32_t spp, uint16_t delay_num, uint16_t delay_den,
                         rt_frame_callback cb, void *user, rt_stats *stats);

/* Count rays the way the reference's work is counted (SURVEY 8d): primary =
 * rows*width*spp^2, shadow = samples with a hit facing the light. */
int rt_count_rays(const rt_scene *s, const rt_camera *camera,
                  uint32_t width, uint32_t height, uint32_t spp,
                  uint32_t row_start, uint32_t row_stride, uint32_t row_count,
                  uint64_t *primary, uint64_t *shadow);

/* Closest-hit traversal of arbitrary rays: TypedGroup::intersect (group.rs:72-83)
 * + Sphere::intersect (primitive.rs:77-84) starting from Hit::missed().  rays and
 * hits are host arrays of n elements. */
int rt_trace_rays(const rt_scene *s, size_t n, const rt_ray *rays, rt_hit *hits);

/* Sustained FP32 FFMA throughput of the scene's device in TFLOP/s, measured with
 * a register-resident FMA chain on every SM (the roofline denominator). */
int rt_measure_fp32_peak(int device, double *tflops, double *sm_clock_mhz);
/* Diagnostics: mode 0 = FFMA chains, mode 1 = alternating FMUL/FADD chains (the
 * unfused mix the parity rule forces on the discriminant), mode 2 = packed FFMA2
 * (sm_100 f32x2), mode 3 = packed FMUL2/FADD2; TFLOP/s counted as 2 flop per FMA
 * and 1 per multiply or add, per component. */
int rt_microbench_fp32(int device, int mode, double *tflops);

/* Diagnostics: compares the kernels' branch-free Newton-step sqrt / reciprocal with
 * the IEEE-rounded intrinsics, and the packed f32x2 versions of sqrt, reciprocal,
 * ray-sphere distance and normalisation with the scalar ones, on n pseudo-random
 * inputs; all six mismatch counters must be 0. */
int rt_selftest_math(uint32_t n, uint32_t seed, uint64_t mismatches[6]);

/* Diagnostics: candidate counts per cull tile of the scene's most recent PHASED frame
 * (counts[2t] = primary, counts[2t+1] = shadow candidates, 0xffffffff = tile rendered by the
 * per-lane walk, 0xfffffffd = shadow rays of the tile all occluded by one leaf, no list and no
 * test); *n_tiles = number of tiles (the capacity of a buffer that only grows: the tiles of the
 * last frame come first), counts may be NULL to query it. */
int rt_debug_phased_tiles(const rt_scene *s, uint32_t cap_tiles, uint32_t *n_tiles, uint32_t *counts);

/* Device memory on the current device, and CUDA IPC handles for it: how the ranks of a
 * multi-process job (one process per GPU) hand rank 0's frame to the others, which then
 * pass `frame + rank*width*4` with pitch `world*width*4` to rt_render_rows -- their kernels
 * store the finished pixels straight into rank 0's HBM over NVLink (no gather step). */
int rt_device_alloc(size_t bytes, void **out);
void rt_device_free(void *p);
int rt_ipc_export(const void *device_ptr, uint8_t handle[64]);
int rt_ipc_open(const uint8_t handle[64], void **out);
int rt_ipc_close(void *p);
/* cudaMemcpy(dst, src, bytes, cudaMemcpyDefault) for buffers obtained above. */
int rt_memcpy(void *dst, const void *src, size_t bytes);
/* cudaMemcpy2DAsync(..., cudaMemcpyDefault, stream): `rows` runs of `width_bytes`, dpitch / spitch apart -- how a
 * rank copies its interleaved row blocks out of a frame-shaped device buffer into a (shared, pinned) host frame. */
int rt_memcpy2d_async(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width_bytes, size_t rows,
                      void *stream);

/* Pinned host memory for output buffers (what the CLI hands to rt_render_frame so
 * the device-to-host copy runs at full PCIe rate).  Replaces the Vec<u8> of
 * RGBABuffer::new (render.rs:80-85). */
int rt_host_alloc(size_t bytes, void **out);
void rt_host_free(void *p);
/* RGBA8 -> RGB8 on the device for the row blocks one GPU owns (blocks of row_block rows at image rows row_start +
 * k * row_stride) of a frame-shaped RGBA buffer, into the same rows of a frame-shaped RGB buffer (width*3 bytes per
 * row): the sink drops alpha anyway (render.rs:389-397), so a rank packs before it copies its blocks out and a
 * quarter of the PCIe traffic is saved.  Rows from `height` on are left untouched.  Asynchronous on `stream`.
 * RT_ERR_INVALID unless both buffers are device memory of the current device, width and height are in 1..65535,
 * 0 < row_block <= row_stride, row_start * width and row_stride * width are multiples of 4 pixels, rgba_frame is
 * 16-byte aligned and rgb_frame 4-byte aligned.  row_start >= height packs nothing and succeeds. */
int rt_pack_rgb_rows(const uint8_t *rgba_frame, uint8_t *rgb_frame, uint32_t width, uint32_t height,
                     uint32_t row_start, uint32_t row_stride, uint32_t row_block, void *stream);
/* Page-lock host memory the caller already owns (e.g. a frame in a shared-memory segment that several
 * processes, one per GPU, copy their row blocks into); portable across devices. */
int rt_host_register(void *p, size_t bytes);
int rt_host_unregister(void *p);
/* Diagnostics: copy-only device-to-host rate (GB/s) of the current device into pinned host memory -- the ceiling of
 * every end-to-end number whose frames leave the GPU; `iters` copies of `bytes` back to back, rotating over
 * `n_buffers` (1..8) host buffers as a sweep's ring of frames does, CUDA events. */
int rt_microbench_d2h(size_t bytes, int iters, int n_buffers, double *gb_per_s);

#ifdef __cplusplus
}
#endif
#endif
