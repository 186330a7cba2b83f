// rt_api.cpp -- the C ABI (include/rtrace.h) over the CUDA kernels.
//
// No torch types, no exceptions across the boundary, no CPU fallback: every
// compute entry point needs a CUDA device and fails with RT_ERR_CUDA otherwise.
#include "../../include/rtrace.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "rt_device.cuh"
#include "rt_kernels.h"
#include "rt_png.h"
#include "rt_scene.h"

namespace {

thread_local char g_err[512] = "";
thread_local int g_variant = RT_VARIANT_AUTO;  // rt_set_variant: the caller's choice for this thread

// How the rows of a launch map to image rows and to rows of the output buffer (rt_render_row_blocks):
// blocks of 2^block_shift consecutive image rows, row_stride apart; out_abs = rows are stored at their
// IMAGE row of a whole frame.  The plain interleave of rt_render_rows is {0, false}.
struct RowLayout {
    uint32_t block_shift = 0;
    bool out_abs = false;
};

// What a sweep hands to its frame callback: the RGBA8 frame, its RGB8 bytes (the P6 body), or a PNG file (with an
// Animation: the frame's payload of an animated PNG).
enum class OutKind { RGBA, RGB, PNG };

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t e_ = (expr);                                                             \
        if (e_ != cudaSuccess) return fail(RT_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

#define RT_TRY(expr)                        \
    do {                                    \
        const int rc_ = (expr);             \
        if (rc_ != RT_OK) return rc_;       \
    } while (0)

// Owners of the CUDA resources a scene (or an encoder's scratch) keeps between calls.  Each releases what it holds
// when it goes, on the current device.
struct NonCopyable {
    NonCopyable() = default;
    NonCopyable(const NonCopyable &) = delete;
    NonCopyable &operator=(const NonCopyable &) = delete;
};

// A grow-only buffer of device memory (Pinned = false) or of pinned, portable host memory (Pinned = true).
template <bool Pinned>
struct Buffer : NonCopyable {
    uint8_t *ptr = nullptr;
    size_t cap = 0;
    ~Buffer() { release(); }
    template <class T>
    T *as() const { return reinterpret_cast<T *>(ptr); }
    // at least `need` bytes; the contents are not kept when the buffer grows
    int ensure(size_t need) {
        if (cap >= need) return RT_OK;
        release();
        cudaError_t e = Pinned ? cudaHostAlloc((void **)&ptr, need, cudaHostAllocPortable) : cudaMalloc((void **)&ptr, need);
        if (e != cudaSuccess) {
            ptr = nullptr;
            return fail(e == cudaErrorMemoryAllocation ? RT_ERR_NOMEM : RT_ERR_CUDA, "%s(%zu): %s",
                        Pinned ? "cudaHostAlloc" : "cudaMalloc", need, cudaGetErrorString(e));
        }
        cap = need;
        return RT_OK;
    }
    void release() {
        if (ptr) Pinned ? cudaFreeHost(ptr) : cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
};
using DeviceBuffer = Buffer<false>;
using HostBuffer = Buffer<true>;

struct Event : NonCopyable {
    cudaEvent_t ev = nullptr;
    ~Event() {
        if (ev) cudaEventDestroy(ev);
    }
    operator cudaEvent_t() const { return ev; }
    int create(unsigned flags) {  // once; later calls keep the event
        if (!ev) CUDA_TRY(cudaEventCreateWithFlags(&ev, flags));
        return RT_OK;
    }
};

// a stream that does not synchronise with the legacy default stream
struct Stream : NonCopyable {
    cudaStream_t st = nullptr;
    ~Stream() {
        if (st) cudaStreamDestroy(st);
    }
    operator cudaStream_t() const { return st; }
    int create() {  // once; later calls keep the stream
        if (!st) CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        return RT_OK;
    }
};

// Scratch of the launches on one stream (launches on different streams may overlap): the PHASED variant's buffers
// and the PNG encoder's.
struct StreamScratch {
    DeviceBuffer winner, hdr, pool, pool_count, png;
    uint32_t pool_units = 0;  // pool entries the kernels may use: a forced RTRACE_POOL_UNITS may leave it below pool.cap
};

// One buffer of the sweep's ring: a frame from its render to its hand-over.
struct SweepSlot {
    DeviceBuffer frame;  // RGBA8
    DeviceBuffer rgb;    // its RGB8 pack (RGB sweeps)
    DeviceBuffer png;    // its PNG file, then the file's length word (PNG sweeps)
    HostBuffer host;     // what the frame callback receives
    HostBuffer len;      // the PNG length word read back
    Event rendered, copied, len_ready;
};

}  // namespace

// ---------------------------------------------------------------------------
// rt_scene
// ---------------------------------------------------------------------------
struct rt_scene {
    int device = 0;
    rt::FlatScene flat;
    uint32_t n = 0;
    DeviceBuffer d_sph, d_skip;  // float4 / uint32_t per node
    // scratch, guarded by mu (a scene may be used from several host threads)
    std::mutex mu;
    DeviceBuffer d_fb, d_kinds;
    DeviceBuffer d_frame;  // gathered frame (multi-GPU root)
    DeviceBuffer d_ctr;    // 16 ray counters
    Event ev0, ev1;
    Stream own_stream;
    // rt_render_sweep: ring of frame buffers (frames rendering at a time + one being copied out), the copy
    // stream and the second render stream
    static constexpr int SWEEP_RING = 3;
    SweepSlot sweep[SWEEP_RING];
    Stream copy_stream, render2;
    std::map<cudaStream_t, StreamScratch> scratch;
    std::mutex mu_scratch;  // guards the map only (mu may already be held by the caller)
};

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// true if ptr is device memory; *dev receives its device ordinal
bool is_device_ptr(const void *ptr, int *dev) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) {
        if (dev) *dev = a.device;
        return true;
    }
    return false;
}

int upload(rt_scene *s) {
    s->n = (uint32_t)s->flat.skip.size();
    CUDA_TRY(cudaGetDevice(&s->device));
    RT_TRY(s->d_sph.ensure(sizeof(float4) * s->n));
    RT_TRY(s->d_skip.ensure(sizeof(uint32_t) * s->n));
    CUDA_TRY(cudaMemcpy(s->d_sph.ptr, s->flat.sph.data(), sizeof(float4) * s->n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(s->d_skip.ptr, s->flat.skip.data(), sizeof(uint32_t) * s->n, cudaMemcpyHostToDevice));
    RT_TRY(s->d_ctr.ensure(sizeof(unsigned long long) * 16));
    RT_TRY(s->ev0.create(cudaEventDefault));
    RT_TRY(s->ev1.create(cudaEventDefault));
    return s->own_stream.create();
}

// The end of both scene constructors: upload the nodes and hand the scene out, or destroy it.
int finish_scene(rt_scene *s, rt_scene **out) {
    const int rc = upload(s);
    if (rc != RT_OK) {
        rt_scene_destroy(s);
        return rc;
    }
    *out = s;
    return RT_OK;
}

void fill_params(const rt_scene *s, const rt_camera *cam, uint32_t w, uint32_t h, uint32_t spp, uint32_t row_start,
                 uint32_t row_stride, uint32_t row_count, rt::RenderParams &p, RowLayout layout = RowLayout()) {
    memset(&p, 0, sizeof(p));
    p.sph = s->d_sph.as<float4>();
    p.skip = s->d_skip.as<uint32_t>();
    p.n_nodes = s->n;
    p.one = 1.0f;
    p.level = s->flat.level;
    p.leaf_rmin = s->flat.leaf_rmin;
    for (int k = 0; k < 3; k++) p.scene_center[k] = s->flat.sph.empty() ? 0.0f : s->flat.sph[k];
    p.scene_radius = s->flat.sph.empty() ? 0.0f : s->flat.sph[3];
    const float *eye = cam ? cam->eye : s->flat.eye;
    for (int k = 0; k < 3; k++) {
        p.eye[k] = eye[k];
        p.light[k] = s->flat.light[k];
    }
    {   // orthonormal pair perpendicular to the light: the plane the shadow pre-filter projects onto
        const double lx = p.light[0], ly = p.light[1], lz = p.light[2];
        const double ln = sqrt(lx * lx + ly * ly + lz * lz);
        if (ln > 0.0) {
            const double l[3] = {lx / ln, ly / ln, lz / ln};
            int m = 0;  // axis least aligned with the light
            if (fabs(l[1]) < fabs(l[m])) m = 1;
            if (fabs(l[2]) < fabs(l[m])) m = 2;
            double a[3] = {0.0, 0.0, 0.0};
            a[m] = 1.0;
            double e1[3] = {l[1] * a[2] - l[2] * a[1], l[2] * a[0] - l[0] * a[2], l[0] * a[1] - l[1] * a[0]};
            const double n1 = sqrt(e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2]);
            for (int k = 0; k < 3; k++) e1[k] /= n1;
            const double e2[3] = {l[1] * e1[2] - l[2] * e1[1], l[2] * e1[0] - l[0] * e1[2], l[0] * e1[1] - l[1] * e1[0]};
            for (int k = 0; k < 3; k++) p.lframe[k] = (float)e1[k], p.lframe[3 + k] = (float)e2[k];
        }
    }
    if (cam) {
        p.has_basis = 1;
        for (int k = 0; k < 3; k++) {
            p.basis[k] = cam->right[k];
            p.basis[3 + k] = cam->up[k];
            p.basis[6 + k] = cam->forward[k];
        }
    }
    p.width = w;
    p.height = h;
    p.spp = spp;
    p.row_start = row_start;
    p.row_stride = row_stride;
    p.row_count = row_count;
    p.row_block_shift = layout.block_shift;
    p.out_abs = layout.out_abs ? 1 : 0;
}

int check_frame_args(const rt_scene *s, uint32_t w, uint32_t h, uint32_t spp, uint32_t row_start, uint32_t row_stride,
                     uint32_t row_count, RowLayout layout = RowLayout()) {
    if (!s) return fail(RT_ERR_INVALID, "scene is NULL");
    // RenderOptions fields are u16 (render.rs:34-38)
    if (w == 0 || h == 0 || w > 65535u || h > 65535u || spp > 65535u)
        return fail(RT_ERR_INVALID, "width/height must be in 1..65535 and samples-per-pixel in 0..65535 (got %u x %u, spp %u)", w, h, spp);
    if (row_stride == 0) return fail(RT_ERR_INVALID, "row_stride must be >= 1");
    if (row_count > 0) {
        const uint32_t j = row_count - 1, bs = layout.block_shift;
        const uint64_t last = (uint64_t)row_start + (uint64_t)(j >> bs) * row_stride + (j & ((1u << bs) - 1u));
        if (last >= h) return fail(RT_ERR_INVALID, "rows starting at %u (stride %u, blocks of %u, %u rows) leave the %u-row image", row_start, row_stride, 1u << bs, row_count, h);
        if (bs && row_stride < (1u << bs)) return fail(RT_ERR_INVALID, "row_stride %u is smaller than the row block %u", row_stride, 1u << bs);
    }
    return RT_OK;
}

// A camera basis must be orthonormal for the TILE variant's cone bounds and PHASED's image-space boxes to hold.
// screen_box (rt_phased.cu) maps a centre into camera space with the basis rows, which inverts the ray rotation
// only up to (B B^T - I) v: row dot products off by 1e-5 move a box by up to ~1 px on a 65535-wide frame and past
// its 0.05 px slack from 4K up.  At 1e-6 every width keeps >= 0.05 px of margin (tests/test_camera_margin.py),
// and a rotation rounded to f32 is off by ~1e-7, so orbit and look-at cameras stay on the fast path.
bool orthonormal(const float b[9]) {
    for (int i = 0; i < 3; i++)
        for (int j = i; j < 3; j++) {
            float d = b[3 * i] * b[3 * j] + b[3 * i + 1] * b[3 * j + 1] + b[3 * i + 2] * b[3 * j + 2];
            if (fabsf(d - (i == j ? 1.0f : 0.0f)) > 1e-6f) return false;
        }
    return true;
}

// AUTO, TILE and PHASED apply to regular pyramids with spp 1..4 and an orthonormal
// camera; anything else falls back to the per-lane walk.  All variants produce
// identical bytes.
// The candidate-list variants compute min over leaves, which equals the reference's pruned
// pre-order walk only while the eye is OUTSIDE every group bound: for an origin inside a bound
// `distance_from_ray` returns the exit distance (primitive.rs:70-71), so `bound >= hit.distance`
// (group.rs:73) may prune a subtree that holds a closer leaf -- an order-dependent result that
// only the per-lane walk reproduces.  All bounds lie inside the root bound, so one test suffices.
bool eye_outside_root_bound(const rt::RenderParams &p) {
    const float dx = p.eye[0] - p.scene_center[0], dy = p.eye[1] - p.scene_center[1], dz = p.eye[2] - p.scene_center[2];
    const float d2 = dx * dx + dy * dy + dz * dz, r = p.scene_radius * 1.0005f + 1e-4f;
    return d2 > r * r;
}

// The conservative pre-filters of TILE / PHASED carry ABSOLUTE slacks (1e-5 on radii, 4e-6 on cone margins,
// 0.05 pixel on image-space boxes) sized for coordinates of magnitude < 16, where one f32 ulp is < 1e-6
// (Scene::default lies within 4.2 of the origin).  A scene or eye placed farther out has coordinate rounding
// above those slacks, so such arguments take the per-lane walk, which has no slack to outgrow.
bool within_analysed_range(const rt::RenderParams &p) {
    float m = 0.0f;
    for (int k = 0; k < 3; k++) m = fmaxf(m, fmaxf(fabsf(p.eye[k]), fabsf(p.scene_center[k]) + p.scene_radius));
    return m <= 16.0f && p.scene_radius > 0.0f;
}

// what the candidate-list variants need beyond their template ranges (rt_tile_supported: spp <= 4,
// rt_phased_supported: spp <= 8; both: regular pyramid of level <= 10)
bool geometry_ok(const rt::RenderParams &p) {
    return (!p.has_basis || orthonormal(p.basis)) && eye_outside_root_bound(p) && within_analysed_range(p);
}

int kernel_variant(const rt::RenderParams &p) {
    if (p.col_count) return g_variant == RT_VARIANT_WARP ? RT_KERNEL_WARP : RT_KERNEL_LANE;  // bucket-sized window
    const bool geo_ok = geometry_ok(p);
    const bool tile_ok = rt_tile_supported(p) && geo_ok, phased_ok = rt_phased_supported(p) && geo_ok;
    switch (g_variant) {
        case RT_VARIANT_LANE:
            return RT_KERNEL_LANE;
        case RT_VARIANT_WARP:
            return RT_KERNEL_WARP;
        case RT_VARIANT_TILE:
            return tile_ok ? RT_KERNEL_TILE : RT_KERNEL_LANE;
        case RT_VARIANT_PHASED:
            return phased_ok ? RT_KERNEL_PHASED : RT_KERNEL_LANE;
        default:
            break;
    }
    if (!phased_ok) return RT_KERNEL_LANE;
    // AUTO (measured on B200, profiles/r01_variant_matrix.json):
    //  * when the smallest leaves project to less than ~1.5 sample spacings the exact test is
    //    rounding noise (SURVEY F3), the cull must inflate them several-fold and the per-lane
    //    walk, which needs no inflation, wins (640x480 level 8: 0.14 vs 0.30 ms);
    //  * frames with few pixel tiles cannot fill the GPU four times over: the fused kernel wins
    //    (1280x720: 0.137 vs 0.147 ms);
    //  * otherwise the four homogeneous launches win (1080p and up, every level <= 10).
    const float dx = p.eye[0] - p.scene_center[0], dy = p.eye[1] - p.scene_center[1], dz = p.eye[2] - p.scene_center[2];
    const float dist = sqrtf(dx * dx + dy * dy + dz * dz);
    const float leaf_px = p.leaf_rmin * (float)p.width / fmaxf(dist, 1e-6f) * (float)p.spp;
    if (leaf_px < 1.5f) return RT_KERNEL_LANE;
    const uint64_t pixel_tiles = (uint64_t)p.width * p.row_count / (p.spp == 1 ? 128u : 32u);  // one warp each
    return (pixel_tiles < 8000 && tile_ok) ? RT_KERNEL_TILE : RT_KERNEL_PHASED;
}

// Float frames have PHASED and LANE kernels only: PHASED wherever RGBA8 would run TILE or PHASED (PHASED is
// correct at every size) and for a forced TILE or PHASED inside PHASED's domain; LANE for everything else,
// including a forced LANE or WARP.
int kernel_variant_f32(const rt::RenderParams &p) {
    switch (g_variant) {
        case RT_VARIANT_LANE:
        case RT_VARIANT_WARP:
            return RT_KERNEL_LANE;
        case RT_VARIANT_TILE:
        case RT_VARIANT_PHASED:
            return rt_phased_supported(p) && geometry_ok(p) ? RT_KERNEL_PHASED : RT_KERNEL_LANE;
        default:
            return kernel_variant(p) == RT_KERNEL_LANE ? RT_KERNEL_LANE : RT_KERNEL_PHASED;
    }
}

// RTRACE_TILE_SHAPE (kernel experiments): the tile shape forced on the TILE and PHASED variants, -1 when unset
int forced_tile_shape() {
    static const char *force = getenv("RTRACE_TILE_SHAPE");
    return (force && *force) ? atoi(force) : -1;
}

// Scratch of the PHASED variant for this stream (allocated on first use, grown on demand).
int prepare_phased(rt_scene *s, rt::RenderParams &p, cudaStream_t stream, int shape) {
    size_t wb = 0, hb = 0;
    uint32_t units = 0;
    rt_phased_scratch(p.width, p.row_count, p.spp, shape, &wb, &hb, &units);
    const char *cap = getenv("RTRACE_POOL_UNITS");  // tests: a tiny pool exercises the overflow fallback
    const bool forced_pool = cap && *cap;
    if (forced_pool) units = (uint32_t)strtoul(cap, nullptr, 10);
    std::lock_guard<std::mutex> lock(s->mu_scratch);
    StreamScratch &sc = s->scratch[stream];
    RT_TRY(sc.winner.ensure(wb));
    RT_TRY(sc.hdr.ensure(hb));
    if (units > sc.pool_units || forced_pool) {  // the pool grows with the frame; only a forced size shrinks it
        sc.pool_units = 0;                          // until the pool holds `units` (a failed ensure frees it)
        RT_TRY(sc.pool.ensure((size_t)units * sizeof(uint4)));
        sc.pool_units = units;
    }
    RT_TRY(sc.pool_count.ensure(sizeof(uint32_t)));
    p.winner = sc.winner.as<uint32_t>();
    p.tile_hdr = sc.hdr.as<uint4>();
    p.pool = sc.pool.as<uint4>();
    p.pool_cap = sc.pool_units;
    p.pool_count = sc.pool_count.as<uint32_t>();
    return RT_OK;
}

// Launches the kernel(s) of one frame on `stream`; *variant receives the kernel that renders it (RT_KERNEL_*,
// numbered like RT_VARIANT_*).
int launch(rt_scene *s, rt::RenderParams &p, bool diag, cudaStream_t stream, int *variant, RtPixels fmt = RT_PIXELS_RGBA8) {
    const int v = fmt == RT_PIXELS_F32 ? kernel_variant_f32(p) : kernel_variant(p), shape = forced_tile_shape();
    *variant = v;
    cudaError_t e;
    if (v == RT_KERNEL_PHASED) {
        const int phased_shape = std::max(shape, 0);
        RT_TRY(prepare_phased(s, p, stream, phased_shape));
        e = rt_launch_render_phased(diag, fmt, p, stream, phased_shape);
    } else if (v == RT_KERNEL_TILE) {
        // AUTO picks the fused kernel only for small frames, where one independent warp per tile
        // (shape 2) beats CTA-shared culls (warps waiting at barriers with too few CTAs to cover them)
        e = rt_launch_render_tile(diag, p, stream, shape >= 0 ? shape : (g_variant == RT_VARIANT_AUTO ? 2 : 0));
    } else {
        e = rt_launch_render(v, diag, fmt, p, stream);
    }
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "kernel launch: %s", cudaGetErrorString(e));
    return RT_OK;
}

uint32_t launches_of(int variant) { return variant == RT_KERNEL_PHASED ? 4 : 1; }

// Queues on `stream` the PNG encode of the RGBA8 frame `rgba` (anim != nullptr: frame `frame`'s payload of that
// animated PNG) into `out` -- the file, then its length word -- and the copy of the length word to *len_host.
// `bound` is the bound of that file (rt_png_bound_bytes).
int queue_encode(const uint8_t *rgba, size_t pitch, uint32_t width, uint32_t height, const Animation *anim,
                 uint32_t frame, size_t bound, DeviceBuffer &scratch, DeviceBuffer &out, unsigned long long *len_host,
                 cudaStream_t stream) {
    const size_t len_at = (bound + 7) / 8 * 8;
    RT_TRY(scratch.ensure(rt_png_scratch_bytes(width, height)));
    RT_TRY(out.ensure(len_at + sizeof(unsigned long long)));
    unsigned long long *len_word = reinterpret_cast<unsigned long long *>(out.ptr + len_at);
    CUDA_TRY(rt_launch_png_encode(rgba, pitch, width, height, anim, frame, scratch.ptr, out.ptr, len_word, stream));
    CUDA_TRY(cudaMemcpyAsync(len_host, len_word, sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
    return RT_OK;
}

// Peer access from device `from` (the current device) to the memory of device `to`: *can = false when there is none.
int enable_peer(int from, int to, bool *can) {
    int c = 0;
    CUDA_TRY(cudaDeviceCanAccessPeer(&c, from, to));
    *can = c != 0;
    if (!c) return RT_OK;
    cudaError_t e = cudaDeviceEnablePeerAccess(to, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(RT_ERR_CUDA, "enable peer access %d->%d: %s", from, to, cudaGetErrorString(e));
    cudaGetLastError();
    return RT_OK;
}

// One replica per GPU: the same scene twice would share one set of scratch buffers and one mutex.
int check_distinct_scenes(rt_scene *const *scenes, int ngpu) {
    std::vector<rt_scene *> order(scenes, scenes + ngpu);
    std::sort(order.begin(), order.end());
    if (std::adjacent_find(order.begin(), order.end()) != order.end())
        return fail(RT_ERR_INVALID, "the same scene was passed twice: one replica per GPU is needed");
    return RT_OK;
}

// rt_encode_png's device buffers for one (device, stream); `mu` serialises the calls that share them.
struct PngEncodeScratch {
    std::mutex mu;
    DeviceBuffer scratch, out;  // out: the file, then its length word
};

}  // namespace

extern "C" {

const char *rt_last_error(void) { return g_err; }
const char *rt_version(void) { return "rtrace-b200 0.2.0 (sm_100a)"; }

int rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int rt_set_device(int device) {
    if (device < 0 || device >= rt_device_count()) return fail(RT_ERR_CUDA, "no CUDA device %d (have %d)", device, rt_device_count());
    CUDA_TRY(cudaSetDevice(device));
    return RT_OK;
}

int rt_set_variant(int variant) {
    if (variant < RT_VARIANT_AUTO || variant > RT_VARIANT_PHASED) return fail(RT_ERR_INVALID, "unknown variant %d", variant);
    g_variant = variant;
    return RT_OK;
}

int rt_scene_create(uint32_t level, const float origin[3], float radius, const float light_unnormalised[3],
                    const float eye[3], rt_scene **out) {
    if (!out || !origin || !light_unnormalised || !eye) return fail(RT_ERR_INVALID, "NULL argument");
    *out = nullptr;
    // group.rs:59-60: "Levels equal or smaller than one cause empty groups"
    if (level <= 1 || level > 12) return fail(RT_ERR_INVALID, "level must be in 2..12 (got %u)", level);
    if (rt_device_count() == 0) return fail(RT_ERR_CUDA, "no CUDA device: librtrace_b200 has no CPU path");
    rt_scene *s = new (std::nothrow) rt_scene();
    if (!s) return fail(RT_ERR_NOMEM, "out of host memory");
    rt::flatten_pyramid(level, origin, radius, s->flat);
    rt::normalize3(light_unnormalised, s->flat.light);
    memcpy(s->flat.eye, eye, sizeof(float) * 3);
    return finish_scene(s, out);
}

int rt_scene_create_default(rt_scene **out) {
    const float origin[3] = {0.0f, -1.0f, 0.0f};  // render.rs:148-152
    const float light[3] = {-1.0f, -3.0f, 2.0f};  // render.rs:154-158
    const float eye[3] = {0.0f, 0.0f, -4.0f};     // render.rs:160-164
    return rt_scene_create(8, origin, 1.0f, light, eye, out);
}

int rt_scene_create_from_nodes(uint32_t n, const float *spheres4, const uint32_t *skip, const float light[3],
                               const float eye[3], rt_scene **out) {
    if (!out || !spheres4 || !skip || !light || !eye) return fail(RT_ERR_INVALID, "NULL argument");
    *out = nullptr;
    uint64_t g = 0, it = 0;
    const char *why = "";
    if (!rt::validate_nodes(n, skip, &g, &it, &why)) return fail(RT_ERR_INVALID, "%s", why);
    if (rt_device_count() == 0) return fail(RT_ERR_CUDA, "no CUDA device: librtrace_b200 has no CPU path");
    rt_scene *s = new (std::nothrow) rt_scene();
    if (!s) return fail(RT_ERR_NOMEM, "out of host memory");
    s->flat.sph.assign(spheres4, spheres4 + (size_t)n * 4);
    s->flat.skip.assign(skip, skip + n);
    s->flat.groups = g;
    s->flat.items = it;
    memcpy(s->flat.light, light, sizeof(float) * 3);
    memcpy(s->flat.eye, eye, sizeof(float) * 3);
    return finish_scene(s, out);
}

void rt_scene_destroy(rt_scene *s) {
    if (!s) return;
    DeviceGuard g(s->device);  // its buffers, events and streams are released on its device
    delete s;
}

int rt_scene_counts(const rt_scene *s, uint64_t *groups, uint64_t *items) {
    if (!s || !groups || !items) return fail(RT_ERR_INVALID, "NULL argument");
    *groups = s->flat.groups;
    *items = s->flat.items;
    return RT_OK;
}

int rt_scene_export_nodes(const rt_scene *s, float *spheres4, uint32_t *skip, uint32_t cap, uint32_t *n_out) {
    if (!s) return fail(RT_ERR_INVALID, "scene is NULL");
    if (n_out) *n_out = s->n;
    if (!spheres4 && !skip) return RT_OK;
    if (cap < s->n) return fail(RT_ERR_BUFFER, "need room for %u nodes, got %u", s->n, cap);
    // read back from the device: this is what the kernels traverse
    DeviceGuard g(s->device);
    if (spheres4) CUDA_TRY(cudaMemcpy(spheres4, s->d_sph.ptr, sizeof(float4) * s->n, cudaMemcpyDeviceToHost));
    if (skip) CUDA_TRY(cudaMemcpy(skip, s->d_skip.ptr, sizeof(uint32_t) * s->n, cudaMemcpyDeviceToHost));
    return RT_OK;
}

int rt_flatten_pyramid_host(uint32_t level, const float origin[3], float radius, float *spheres4, uint32_t *skip,
                            uint32_t cap, uint32_t *n_out) {
    if (!origin) return fail(RT_ERR_INVALID, "NULL argument");
    if (level <= 1 || level > 12) return fail(RT_ERR_INVALID, "level must be in 2..12 (got %u)", level);
    const uint32_t n = (uint32_t)rt::pyramid_subtree_nodes(level);
    if (n_out) *n_out = n;
    if (!spheres4 && !skip) return RT_OK;
    if (cap < n) return fail(RT_ERR_BUFFER, "need room for %u nodes, got %u", n, cap);
    rt::FlatScene f;
    rt::flatten_pyramid(level, origin, radius, f);
    if (spheres4) memcpy(spheres4, f.sph.data(), sizeof(float) * 4 * n);
    if (skip) memcpy(skip, f.skip.data(), sizeof(uint32_t) * n);
    return RT_OK;
}

int rt_scene_light(const rt_scene *s, float light[3]) {
    if (!s || !light) return fail(RT_ERR_INVALID, "NULL argument");
    memcpy(light, s->flat.light, sizeof(float) * 3);
    return RT_OK;
}

int rt_scene_eye(const rt_scene *s, float eye[3]) {
    if (!s || !eye) return fail(RT_ERR_INVALID, "NULL argument");
    memcpy(eye, s->flat.eye, sizeof(float) * 3);
    return RT_OK;
}

int rt_scene_device(const rt_scene *s) { return s ? s->device : fail(RT_ERR_INVALID, "scene is NULL"); }

// ---------------------------------------------------------------------------
// hot path
// ---------------------------------------------------------------------------
static int render_rows_impl(rt_scene *s, const rt_camera *camera, uint32_t width, uint32_t height, uint32_t spp,
                            uint32_t row_start, uint32_t row_stride, uint32_t row_count, uint8_t *rgba_out,
                            size_t pitch_bytes, uint8_t *kinds_out, cudaStream_t stream, rt_stats *stats,
                            uint64_t *count_hits, uint64_t *count_shadow, uint32_t col_start = 0,
                            uint32_t col_count = 0, RowLayout layout = RowLayout(), RtPixels fmt = RT_PIXELS_RGBA8) {
    int rc = check_frame_args(s, width, height, spp, row_start, row_stride, row_count, layout);
    if (rc != RT_OK) return rc;
    const bool counting = count_shadow != nullptr;
    if (!rgba_out && !counting) return fail(RT_ERR_INVALID, "rgba_out is NULL");
    // col_count > 0: only columns col_start .. col_start + col_count - 1, packed from byte 0 of each output row
    if ((uint64_t)col_start + col_count > width) return fail(RT_ERR_INVALID, "columns %u..%u leave the %u-pixel row", col_start, col_start + col_count, width);
    const uint32_t cols = col_count ? col_count : width;
    const size_t bpp = fmt == RT_PIXELS_F32 ? 16 : 4;  // bytes per pixel; pitches and device pointers are multiples of it
    const size_t row_bytes = (size_t)cols * bpp;
    if (pitch_bytes == 0) pitch_bytes = row_bytes;
    if (pitch_bytes < row_bytes || (pitch_bytes & (bpp - 1))) return fail(RT_ERR_INVALID, "pitch %zu too small or not a multiple of %zu", pitch_bytes, bpp);
    if (stats) memset(stats, 0, sizeof(*stats));
    if (row_count == 0) return RT_OK;

    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(RT_ERR_CUDA, "cannot select device %d", s->device);
    const double t0 = now_ms();

    int out_dev = -1;
    const bool out_on_device = rgba_out && is_device_ptr(rgba_out, &out_dev);
    if (out_on_device && out_dev != s->device) {
        // a peer GPU's memory (e.g. rank 0's frame): the kernel stores over NVLink
        bool can = false;
        RT_TRY(enable_peer(s->device, out_dev, &can));
        if (!can) return fail(RT_ERR_INVALID, "rgba_out lives on device %d, which device %d cannot access", out_dev, s->device);
    }
    if (out_on_device && (((uintptr_t)rgba_out) & (bpp - 1))) return fail(RT_ERR_INVALID, "device rgba_out must be %zu-byte aligned", bpp);
    int kinds_dev = -1;
    const bool kinds_on_device = kinds_out && is_device_ptr(kinds_out, &kinds_dev);
    const size_t kinds_bytes = (size_t)cols * row_count * spp * spp;

    if (layout.out_abs && !out_on_device) return fail(RT_ERR_INVALID, "absolute row addressing needs a device (or peer) frame buffer");
    const bool need_lock = !out_on_device || (kinds_out && !kinds_on_device) || counting || stats;
    std::unique_lock<std::mutex> lock(s->mu, std::defer_lock);
    if (need_lock) lock.lock();

    rt::RenderParams p;
    fill_params(s, camera, width, height, spp, row_start, row_stride, row_count, p, layout);
    p.col_start = col_count ? col_start : 0;
    p.col_count = col_count;
    if (out_on_device) {
        p.out = rgba_out;
        p.pitch = pitch_bytes;
    } else {
        RT_TRY(s->d_fb.ensure(row_bytes * row_count));
        p.out = s->d_fb.ptr;
        p.pitch = row_bytes;
    }
    bool diag = false;
    if (kinds_out) {
        diag = true;
        if (kinds_on_device) {
            p.kinds = kinds_out;
        } else {
            RT_TRY(s->d_kinds.ensure(kinds_bytes ? kinds_bytes : 1));
            p.kinds = s->d_kinds.ptr;
        }
    }
    if (counting) {
        diag = true;
        p.ray_counters = s->d_ctr.as<unsigned long long>();
        CUDA_TRY(cudaMemsetAsync(s->d_ctr.ptr, 0, sizeof(unsigned long long) * 16, stream));
    }

    if (stats) CUDA_TRY(cudaEventRecord(s->ev0, stream));
    int variant = 0;
    RT_TRY(launch(s, p, diag, stream, &variant, fmt));
    if (stats) CUDA_TRY(cudaEventRecord(s->ev1, stream));

    bool must_sync = false;
    if (!out_on_device && rgba_out) {
        CUDA_TRY(cudaMemcpy2DAsync(rgba_out, pitch_bytes, s->d_fb.ptr, row_bytes, row_bytes, row_count, cudaMemcpyDeviceToHost, stream));
        must_sync = true;
    }
    if (kinds_out && !kinds_on_device && kinds_bytes) {
        CUDA_TRY(cudaMemcpyAsync(kinds_out, s->d_kinds.ptr, kinds_bytes, cudaMemcpyDeviceToHost, stream));
        must_sync = true;
    }
    unsigned long long ctr[16] = {0};
    if (counting) {
        CUDA_TRY(cudaMemcpyAsync(ctr, s->d_ctr.ptr, sizeof(ctr), cudaMemcpyDeviceToHost, stream));
        must_sync = true;
    }
    if (must_sync || stats) CUDA_TRY(cudaStreamSynchronize(stream));
    if (counting) {
        if (count_hits) *count_hits = ctr[0];
        *count_shadow = ctr[1];
        if (getenv("RTRACE_PROFILE")) {  // phase totals of an -DRT_TILE_PROFILE build
            fprintf(stderr, "rt-profile:");
            for (int k = 2; k < 16; k++) fprintf(stderr, " %llu", ctr[k]);
            fprintf(stderr, "\n");
        }
    }
    if (stats) {
        float ms = 0.0f;
        CUDA_TRY(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
        stats->kernel_ms = ms;
        stats->total_ms = now_ms() - t0;
        stats->primary_rays = (uint64_t)cols * row_count * spp * spp;
        stats->shadow_rays = counting ? ctr[1] : 0;
        stats->kernel_launches = launches_of(variant);
        stats->gpus = 1;
        stats->variant_used = (uint32_t)variant;
    }
    return RT_OK;
}

int rt_render_rows(const rt_scene *s, const rt_camera *camera, uint32_t width, uint32_t height, uint32_t spp,
                   uint32_t row_start, uint32_t row_stride, uint32_t row_count, uint8_t *rgba_out, size_t pitch_bytes,
                   uint8_t *kinds_out, void *stream, rt_stats *stats) {
    return render_rows_impl(const_cast<rt_scene *>(s), camera, width, height, spp, row_start, row_stride, row_count,
                            rgba_out, pitch_bytes, kinds_out, (cudaStream_t)stream, stats, nullptr, nullptr);
}

int rt_render_rows_f32(const rt_scene *s, const rt_camera *camera, uint32_t width, uint32_t height, uint32_t spp,
                       uint32_t row_start, uint32_t row_stride, uint32_t row_count, float *rgba_out, size_t pitch_bytes,
                       void *stream, rt_stats *stats) {
    if (!rgba_out) return fail(RT_ERR_INVALID, "rgba_out is NULL");
    return render_rows_impl(const_cast<rt_scene *>(s), camera, width, height, spp, row_start, row_stride, row_count,
                            reinterpret_cast<uint8_t *>(rgba_out), pitch_bytes, nullptr, (cudaStream_t)stream, stats,
                            nullptr, nullptr, 0, 0, RowLayout(), RT_PIXELS_F32);
}

int rt_render_row_blocks(const rt_scene *s, const rt_camera *camera, uint32_t width, uint32_t height, uint32_t spp,
                         uint32_t row_start, uint32_t row_stride, uint32_t row_block, uint32_t row_count, uint8_t *rgba_out,
                         size_t pitch_bytes, int absolute_rows, void *stream, rt_stats *stats) {
    if (row_block == 0 || (row_block & (row_block - 1u)) || row_block > 32768u) return fail(RT_ERR_INVALID, "row_block must be a power of two (got %u)", row_block);
    uint32_t shift = 0;
    while ((1u << shift) < row_block) shift++;
    RowLayout layout;
    layout.block_shift = shift;
    layout.out_abs = absolute_rows != 0;
    return render_rows_impl(const_cast<rt_scene *>(s), camera, width, height, spp, row_start, row_stride, row_count,
                            rgba_out, pitch_bytes, nullptr, (cudaStream_t)stream, stats, nullptr, nullptr, 0, 0, layout);
}

int rt_render_region(const rt_scene *s, uint16_t width, uint16_t height, uint16_t spp, uint16_t l, uint16_t b,
                     uint16_t r, uint16_t t, uint8_t *rgba_out, size_t rgba_len) {
    if (!s) return fail(RT_ERR_INVALID, "scene is NULL");
    // ImageRegion (render.rs:43-72): l <= r <= width, b <= t <= height
    if (l > r || b > t || r > width || t > height)
        return fail(RT_ERR_INVALID, "region [%u,%u)x[%u,%u) is not inside the %ux%u image", l, r, b, t, width, height);
    const uint32_t rw = r - l, rh = t - b;
    if (rgba_len < (size_t)rw * rh * 4) return fail(RT_ERR_BUFFER, "rgba_out holds %zu bytes, region needs %zu", rgba_len, (size_t)rw * rh * 4);
    if (rw == 0 || rh == 0) return RT_OK;
    if (l == 0 && r == width)
        return render_rows_impl(const_cast<rt_scene *>(s), nullptr, width, height, spp, b, 1, rh, rgba_out, 0, nullptr,
                                nullptr, nullptr, nullptr, nullptr);
    // A bucket (render.rs:273-298 cuts the frame into 64x64 of them): the per-lane kernel renders just the
    // window, so the cost of a region is proportional to its area.
    return render_rows_impl(const_cast<rt_scene *>(s), nullptr, width, height, spp, b, 1, rh, rgba_out, 0, nullptr,
                            nullptr, nullptr, nullptr, nullptr, l, rw);
}

int rt_render_frame(const rt_scene *s, const rt_camera *camera, uint32_t width, uint32_t height, uint32_t spp,
                    uint8_t *rgba_out, size_t rgba_len, rt_stats *stats) {
    if (rgba_len < (size_t)width * height * 4) return fail(RT_ERR_BUFFER, "rgba_out holds %zu bytes, frame needs %zu", rgba_len, (size_t)width * height * 4);
    return render_rows_impl(const_cast<rt_scene *>(s), camera, width, height, spp, 0, 1, height, rgba_out, 0, nullptr,
                            nullptr, stats, nullptr, nullptr);
}

int rt_render_preview(const rt_scene *cs, const rt_camera *camera, uint32_t width, uint32_t height, uint32_t step,
                      uint8_t *rgba_out, size_t rgba_len, void *stream_) {
    rt_scene *s = const_cast<rt_scene *>(cs);
    cudaStream_t stream = (cudaStream_t)stream_;
    if (step == 0 || step > 1024u) return fail(RT_ERR_INVALID, "step must be in 1..1024 (got %u)", step);
    int rc = check_frame_args(s, width, height, 1, 0, 1, height);
    if (rc != RT_OK) return rc;
    if (!rgba_out) return fail(RT_ERR_INVALID, "rgba_out is NULL");
    const size_t row_bytes = (size_t)width * 4, frame_bytes = row_bytes * height;
    if (rgba_len < frame_bytes) return fail(RT_ERR_BUFFER, "rgba_out holds %zu bytes, frame needs %zu", rgba_len, frame_bytes);
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(RT_ERR_CUDA, "cannot select device %d", s->device);
    int out_dev = -1;
    const bool out_on_device = is_device_ptr(rgba_out, &out_dev);
    if (out_on_device && out_dev != s->device) return fail(RT_ERR_INVALID, "rgba_out lives on device %d, the scene on device %d", out_dev, s->device);
    if (out_on_device && (((uintptr_t)rgba_out) & 3)) return fail(RT_ERR_INVALID, "device rgba_out must be 4-byte aligned");
    std::unique_lock<std::mutex> lock(s->mu, std::defer_lock);
    if (!out_on_device) lock.lock();  // the staging frame is per scene
    rt::RenderParams p;
    const uint32_t bx = (width + step - 1) / step, by = (height + step - 1) / step;  // blocks = traced pixels
    fill_params(s, camera, width, height, 1, 0, 1, by, p);
    p.col_count = bx;
    p.px_step = step;
    p.pitch = row_bytes;
    if (out_on_device) {
        p.out = rgba_out;
    } else {
        RT_TRY(s->d_fb.ensure(frame_bytes));
        p.out = s->d_fb.ptr;
    }
    cudaError_t e = rt_launch_render_preview(p, stream);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "kernel launch: %s", cudaGetErrorString(e));
    if (!out_on_device) {
        CUDA_TRY(cudaMemcpyAsync(rgba_out, s->d_fb.ptr, frame_bytes, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
    }
    return RT_OK;
}

// Where a sweep's frames come from: called when the pipeline has room for another frame; returns its id (>= 0, handed
// back to the frame callback) and fills *cam (use_cam = false: the reference camera), or -1 when there is none left.
struct FrameSource {
    virtual ~FrameSource() {}
    virtual int64_t next(rt_camera *cam, bool *use_cam) = 0;
};

// cameras[0 .. n): the fixed list of rt_render_sweep
struct ListSource : FrameSource {
    const rt_camera *cameras;
    uint32_t n, at = 0;
    ListSource(const rt_camera *c, uint32_t n_) : cameras(c), n(n_) {}
    int64_t next(rt_camera *cam, bool *use_cam) override {
        if (at >= n) return -1;
        *use_cam = cameras != nullptr;
        if (cameras) *cam = cameras[at];
        return (int64_t)at++;
    }
};

// the caller's rt_next_frame_callback (rt_render_sweep_pull)
struct CallbackSource : FrameSource {
    rt_next_frame_callback fn;
    void *user;
    CallbackSource(rt_next_frame_callback f, void *u) : fn(f), user(u) {}
    int64_t next(rt_camera *cam, bool *use_cam) override {
        int use = 1;
        const int64_t id = fn ? (int64_t)fn(user, cam, &use) : -1;
        *use_cam = use != 0;
        return id;
    }
};

static int sweep_locked(rt_scene *s, FrameSource &src, uint32_t width, uint32_t height, uint32_t spp, rt_frame_callback cb,
                        void *user, rt_stats *stats, OutKind kind, const Animation *anim);

static int sweep_impl(const rt_scene *cs, FrameSource &src, uint32_t width, uint32_t height, uint32_t spp,
                      rt_frame_callback cb, void *user, rt_stats *stats, OutKind kind, const Animation *anim = nullptr) {
    rt_scene *s = const_cast<rt_scene *>(cs);
    int rc = check_frame_args(s, width, height, spp, 0, 1, height);
    if (rc != RT_OK) return rc;
    if (stats) memset(stats, 0, sizeof(*stats));
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(RT_ERR_CUDA, "cannot select device %d", s->device);
    std::lock_guard<std::mutex> lock(s->mu);
    rc = sweep_locked(s, src, width, height, spp, cb, user, stats, kind, anim);
    if (rc != RT_OK) {  // leave no render or copy in flight on the ring buffers (keeps the first error text)
        if (s->own_stream) cudaStreamSynchronize(s->own_stream);
        if (s->render2) cudaStreamSynchronize(s->render2);
        if (s->copy_stream) cudaStreamSynchronize(s->copy_stream);
        cudaGetLastError();
    }
    return rc;
}

// anim != nullptr (PNG only): every frame is its payload of that animated PNG
static int sweep_locked(rt_scene *s, FrameSource &src, uint32_t width, uint32_t height, uint32_t spp, rt_frame_callback cb,
                        void *user, rt_stats *stats, OutKind kind, const Animation *anim) {
    const double t0 = now_ms();
    const bool rgb = kind == OutKind::RGB, png = kind == OutKind::PNG;
    const size_t row_bytes = (size_t)width * 4, frame_bytes = row_bytes * height;
    const size_t out_bytes = rgb ? (size_t)width * height * 3 : frame_bytes;
    const size_t png_bytes = png ? rt_png_bound_bytes(width, height, anim) : 0;
    const size_t host_bytes = std::max(frame_bytes, png_bytes);
    // `depth` frames render at a time, each on its own stream (depth 2: the launch tails of frame f are filled
    // by the first launches of frame f+1), while an earlier frame is copied out: depth + 1 device frames and
    // pinned host frames.  Measured on B200 (C5, 4K 4x4 level 9): 1.395 ms per delivered frame with one render
    // stream, 1.294 ms with two -- less than a lone frame's 1.34 ms of kernels.  RTRACE_SWEEP_STREAMS=1 selects
    // the single-stream schedule (kernel experiments).
    int depth = 2;
    if (const char *e = getenv("RTRACE_SWEEP_STREAMS")) {
        if (*e == '1') depth = 1;
    }
    const int nb = depth + 1;
    if (depth == 2) RT_TRY(s->render2.create());
    RT_TRY(s->copy_stream.create());
    uint32_t launches = 0, used = 0;
    uint64_t issued = 0, delivered = 0;  // frames put into / handed out of the ring, in this order
    int64_t ids[rt_scene::SWEEP_RING] = {0, 0, 0};
    bool more = true;
    while (more || delivered < issued) {
        if (more) {  // the ring has room (a frame is delivered below whenever `depth` are in flight): take the next frame
            rt_camera cam;
            bool use_cam = false;
            const int64_t id = src.next(&cam, &use_cam);
            if (id < 0) {
                more = false;
            } else {
                const int k = (int)(issued % (uint64_t)nb);
                SweepSlot &sl = s->sweep[k];
                ids[k] = id;
                RT_TRY(sl.frame.ensure(frame_bytes));
                RT_TRY(sl.host.ensure(host_bytes));
                if (rgb) RT_TRY(sl.rgb.ensure(frame_bytes / 4 * 3 + 16));
                if (png) RT_TRY(sl.len.ensure(sizeof(unsigned long long)));
                for (Event *e : {&sl.rendered, &sl.copied, &sl.len_ready}) RT_TRY(e->create(cudaEventDisableTiming));
                cudaStream_t rs = (depth == 2 && (issued & 1u)) ? s->render2 : s->own_stream;  // PHASED scratch is per stream
                rt::RenderParams p;
                fill_params(s, use_cam ? &cam : nullptr, width, height, spp, 0, 1, height, p);
                p.out = sl.frame.ptr;
                p.pitch = row_bytes;
                if (issued >= (uint64_t)nb) CUDA_TRY(cudaStreamWaitEvent(rs, sl.copied, 0));  // its previous frame has left this buffer
                int variant = 0;
                RT_TRY(launch(s, p, false, rs, &variant));
                launches += launches_of(variant);
                used = (uint32_t)variant;
                if (rgb) {  // the sink only needs RGB: pack on the device, copy 3 bytes per pixel
                    CUDA_TRY(rt_launch_pack_rgb(sl.frame.ptr, sl.rgb.ptr, (size_t)width * height, rs));
                    launches += 1;
                }
                if (png) {
                    // encode behind the frame's launches; only the length word comes back now (on the render
                    // stream, so that the copy stream never waits for a later frame); the file is copied at hand-over
                    {
                        std::lock_guard<std::mutex> lock(s->mu_scratch);
                        RT_TRY(queue_encode(sl.frame.ptr, row_bytes, width, height, anim, (uint32_t)id, png_bytes,
                                            s->scratch[rs].png, sl.png, sl.len.as<unsigned long long>(), rs));
                    }
                    CUDA_TRY(cudaEventRecord(sl.len_ready, rs));
                    launches += 2;
                } else {
                    CUDA_TRY(cudaEventRecord(sl.rendered, rs));
                    CUDA_TRY(cudaStreamWaitEvent(s->copy_stream, sl.rendered, 0));
                    CUDA_TRY(cudaMemcpyAsync(sl.host.ptr, rgb ? sl.rgb.ptr : sl.frame.ptr, out_bytes, cudaMemcpyDeviceToHost, s->copy_stream));
                    CUDA_TRY(cudaEventRecord(sl.copied, s->copy_stream));
                }
                issued++;
            }
        }
        if (issued - delivered > (uint64_t)depth || (!more && delivered < issued)) {
            // hand the oldest frame to the caller while the later ones render
            const int k = (int)(delivered % (uint64_t)nb);
            SweepSlot &sl = s->sweep[k];
            size_t len = out_bytes;
            if (png) {  // the file's length first, then just that many bytes
                CUDA_TRY(cudaEventSynchronize(sl.len_ready));
                len = (size_t)*sl.len.as<unsigned long long>();
                if (len > png_bytes) return fail(RT_ERR_CUDA, "PNG encoder returned %zu bytes, more than the bound %zu", len, png_bytes);
                CUDA_TRY(cudaMemcpyAsync(sl.host.ptr, sl.png.ptr, len, cudaMemcpyDeviceToHost, s->copy_stream));
                CUDA_TRY(cudaEventRecord(sl.copied, s->copy_stream));
            }
            CUDA_TRY(cudaEventSynchronize(sl.copied));
            if (cb) cb(user, (uint32_t)ids[k], sl.host.ptr, len);
            delivered++;
        }
    }
    if (stats) {
        stats->total_ms = now_ms() - t0;
        stats->primary_rays = (uint64_t)width * height * spp * spp * issued;
        stats->kernel_launches = launches;
        stats->gpus = 1;
        stats->variant_used = used;
    }
    return RT_OK;
}

int rt_render_sweep(const rt_scene *s, const rt_camera *cameras, uint32_t n_frames, uint32_t width, uint32_t height,
                    uint32_t spp, rt_frame_callback cb, void *user, rt_stats *stats) {
    ListSource src(cameras, n_frames);
    return sweep_impl(s, src, width, height, spp, cb, user, stats, OutKind::RGBA);
}

int rt_render_sweep_rgb(const rt_scene *s, const rt_camera *cameras, uint32_t n_frames, uint32_t width, uint32_t height,
                        uint32_t spp, rt_frame_callback cb, void *user, rt_stats *stats) {
    ListSource src(cameras, n_frames);
    return sweep_impl(s, src, width, height, spp, cb, user, stats, OutKind::RGB);
}

int rt_render_sweep_pull(const rt_scene *s, rt_next_frame_callback next, void *next_user, uint32_t width, uint32_t height,
                         uint32_t spp, int rgb, rt_frame_callback cb, void *user, rt_stats *stats) {
    if (!next) return fail(RT_ERR_INVALID, "next-frame callback is NULL");
    CallbackSource src(next, next_user);
    return sweep_impl(s, src, width, height, spp, cb, user, stats, rgb ? OutKind::RGB : OutKind::RGBA);
}

// Body of rt_render_frame_multi once every scene's scratch is locked.  `launched` records the GPUs that have
// work in flight, so that the caller can drain them whatever happens here.
//
// GPU g renders blocks of 16 consecutive rows, G blocks apart (whole cull tiles stay contiguous in the image).
//  * HOST output (the CLI's sink): every GPU renders its blocks at their image rows of its OWN frame buffer and
//    then copies just those blocks to the caller's buffer over its own PCIe link (one strided copy per GPU, all
//    links in parallel).  Nothing is gathered on a GPU: the host frame is where the bands meet.  An 8K RGBA
//    frame is 133 MB -- 2.5 ms over one link, against 0.7 ms of rendering on 8 GPUs.
//  * DEVICE output (a frame on GPU 0, e.g. for a device-side consumer): the kernels of GPU g > 0 store their
//    pixels straight into that frame through peer memory over NVLink -- the stores are the gather.  Without
//    peer access GPU g renders rows g, g+G, ... into a band of its own and a strided peer copy de-interleaves it.
static int frame_multi_locked(rt_scene *const *scenes, int ngpu, const rt_camera *camera, uint32_t width, uint32_t height,
                              uint32_t spp, uint8_t *rgba_out, rt_stats *stats, std::vector<char> &launched,
                              RtPixels fmt) {
    const double t0 = now_ms();
    const size_t row_bytes = (size_t)width * (fmt == RT_PIXELS_F32 ? 16 : 4);
    rt_scene *root = scenes[0];
    int out_dev = -1;
    const bool to_device = is_device_ptr(rgba_out, &out_dev);
    if (to_device && out_dev != root->device) return fail(RT_ERR_INVALID, "a device rgba_out must live on the first scene's GPU (%d), not %d", root->device, out_dev);
    uint8_t *frame = to_device ? rgba_out : nullptr;  // the gathered device frame (device output only)
    uint32_t launches = 0, used = 0;
    const uint32_t B = 16;
    for (int g = 0; g < ngpu; g++) {
        rt_scene *s = scenes[g];
        DeviceGuard guard(s->device);
        if (!guard.ok) return fail(RT_ERR_CUDA, "cannot select device %d", s->device);
        bool peer = g == 0 || !to_device;
        if (!peer) RT_TRY(enable_peer(s->device, root->device, &peer));
        rt::RenderParams p;
        uint32_t rows;
        const uint32_t first = (uint32_t)g * B, stride = (uint32_t)ngpu * B;
        if (peer) {
            rows = 0;
            for (uint64_t y0 = first; y0 < height; y0 += stride) rows += (uint32_t)std::min<uint64_t>(B, height - y0);
            if (rows == 0) continue;
            RowLayout layout;
            layout.block_shift = 4;
            layout.out_abs = true;
            fill_params(s, camera, width, height, spp, first, stride, rows, p, layout);
            if (to_device) {
                p.out = frame;
            } else {
                RT_TRY(s->d_frame.ensure(row_bytes * height));
                p.out = s->d_frame.ptr;
            }
            p.pitch = row_bytes;
        } else {
            rows = (height > (uint32_t)g) ? (height - g + ngpu - 1) / ngpu : 0;
            if (rows == 0) continue;
            fill_params(s, camera, width, height, spp, (uint32_t)g, (uint32_t)ngpu, rows, p);
            RT_TRY(s->d_fb.ensure(row_bytes * rows));
            p.out = s->d_fb.ptr;
            p.pitch = row_bytes;
        }
        if (stats) CUDA_TRY(cudaEventRecord(s->ev0, s->own_stream));
        launched[(size_t)g] = 1;  // from here on this GPU may have work in flight
        int variant = 0;
        RT_TRY(launch(s, p, false, s->own_stream, &variant, fmt));
        launches += launches_of(variant);
        if (g == 0) used = (uint32_t)variant;
        if (stats) CUDA_TRY(cudaEventRecord(s->ev1, s->own_stream));
        if (!to_device) {
            // this GPU's blocks -> the host frame: whole blocks as one strided copy, then the partial last block
            const size_t blk = (size_t)B * row_bytes, pitch = (size_t)stride * row_bytes, off = (size_t)first * row_bytes;
            const uint32_t whole = rows / B, tail = rows % B;
            if (whole) CUDA_TRY(cudaMemcpy2DAsync(rgba_out + off, pitch, s->d_frame.ptr + off, pitch, blk, whole, cudaMemcpyDeviceToHost, s->own_stream));
            if (tail) CUDA_TRY(cudaMemcpyAsync(rgba_out + off + (size_t)whole * pitch, s->d_frame.ptr + off + (size_t)whole * pitch, (size_t)tail * row_bytes, cudaMemcpyDeviceToHost, s->own_stream));
        } else if (!peer) {  // no peer access: strided copy, the pitch de-interleaves the band into the frame
            CUDA_TRY(cudaMemcpy2DAsync(frame + row_bytes * g, row_bytes * ngpu, s->d_fb.ptr, row_bytes, row_bytes, rows, cudaMemcpyDefault, s->own_stream));
        }
    }
    double kmax = 0.0;
    for (int g = ngpu - 1; g >= 0; g--) {
        rt_scene *s = scenes[g];
        DeviceGuard guard(s->device);
        CUDA_TRY(cudaStreamSynchronize(s->own_stream));
        if (stats && launched[(size_t)g]) {
            float ms = 0.0f;
            CUDA_TRY(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
            if (ms > kmax) kmax = ms;
        }
    }
    if (stats) {
        stats->kernel_ms = kmax;
        stats->total_ms = now_ms() - t0;
        stats->primary_rays = (uint64_t)width * height * spp * spp;
        stats->kernel_launches = launches;
        stats->gpus = (uint32_t)ngpu;
        stats->variant_used = used;
    }
    return RT_OK;
}

// Distinct scenes, locked in address order (two threads passing the same scenes in different orders cannot
// deadlock).
static int lock_scenes(rt_scene *const *scenes, int ngpu, std::vector<std::unique_lock<std::mutex>> &locks) {
    RT_TRY(check_distinct_scenes(scenes, ngpu));
    std::vector<rt_scene *> order(scenes, scenes + ngpu);
    std::sort(order.begin(), order.end());
    for (rt_scene *s : order) locks.emplace_back(s->mu);
    return RT_OK;
}

// rt_render_frame_multi and rt_render_frame_multi_f32: the frame at 4 or 16 bytes per pixel.
static int frame_multi_impl(rt_scene *const *scenes, int ngpu, const rt_camera *camera, uint32_t width, uint32_t height,
                            uint32_t spp, uint8_t *rgba_out, size_t rgba_len, rt_stats *stats, RtPixels fmt) {
    if (!scenes || ngpu < 1) return fail(RT_ERR_INVALID, "need at least one scene");
    if (!rgba_out) return fail(RT_ERR_INVALID, "rgba_out is NULL");
    const size_t bpp = fmt == RT_PIXELS_F32 ? 16 : 4, frame_bytes = (size_t)width * height * bpp;
    if (rgba_len < frame_bytes) return fail(RT_ERR_BUFFER, "rgba_out holds %zu bytes, frame needs %zu", rgba_len, frame_bytes);
    for (int g = 0; g < ngpu; g++) {
        int rc = check_frame_args(scenes[g], width, height, spp, 0, 1, height);
        if (rc != RT_OK) return rc;
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    if (ngpu == 1)
        return render_rows_impl(scenes[0], camera, width, height, spp, 0, 1, height, rgba_out, 0, nullptr, nullptr,
                                stats, nullptr, nullptr, 0, 0, RowLayout(), fmt);
    if (fmt == RT_PIXELS_F32 && is_device_ptr(rgba_out, nullptr) && ((uintptr_t)rgba_out & 15))
        return fail(RT_ERR_INVALID, "device rgba_out must be 16-byte aligned");

    std::vector<std::unique_lock<std::mutex>> locks;
    int rc = lock_scenes(scenes, ngpu, locks);
    if (rc != RT_OK) return rc;
    std::vector<char> launched((size_t)ngpu, 0);  // GPUs whose share of the rows is not empty
    rc = frame_multi_locked(scenes, ngpu, camera, width, height, spp, rgba_out, stats, launched, fmt);
    if (rc != RT_OK) {
        // Kernels already launched on other GPUs may still be storing into GPU 0's frame through peer memory:
        // drain every GPU before the locks are released (a later call may free or reuse that frame).  Keeps
        // the first error text.
        for (int g = 0; g < ngpu; g++) {
            if (!launched[(size_t)g]) continue;
            DeviceGuard guard(scenes[g]->device);
            cudaStreamSynchronize(scenes[g]->own_stream);
        }
        cudaGetLastError();
    }
    return rc;
}

int rt_render_frame_multi(rt_scene *const *scenes, int ngpu, const rt_camera *camera, uint32_t width, uint32_t height,
                          uint32_t spp, uint8_t *rgba_out, size_t rgba_len, rt_stats *stats) {
    return frame_multi_impl(scenes, ngpu, camera, width, height, spp, rgba_out, rgba_len, stats, RT_PIXELS_RGBA8);
}

int rt_render_frame_multi_f32(rt_scene *const *scenes, int ngpu, const rt_camera *camera, uint32_t width, uint32_t height,
                              uint32_t spp, float *rgba_out, size_t rgba_bytes, rt_stats *stats) {
    return frame_multi_impl(scenes, ngpu, camera, width, height, spp, reinterpret_cast<uint8_t *>(rgba_out), rgba_bytes,
                            stats, RT_PIXELS_F32);
}

// ---------------------------------------------------------------------------
// Frame-sharded sweep over the GPUs of this process (BASELINE configs[4])
// ---------------------------------------------------------------------------
// The reference has ONE scheduler that owns every unit of work and a consumer that takes the results as they
// come (render.rs:271-307: pool.execute per bucket, sync_channel(4), the main thread draining into the
// writer).  Here the unit is a frame and the pool is the GPUs: every GPU runs the pipelined single-GPU sweep on
// its own host thread and PULLS the next frame of the list whenever its pipeline has room, so a GPU whose host
// link is slower (on the 8-GPU boxes of this pool four GPUs share one uplink: 12.6 GB/s each under load against
// 21 GB/s for the other four) simply takes fewer frames.  The calling thread hands the frames to `cb` in frame
// order; a worker whose frame is not yet due blocks in its hand-over (its pinned buffer is only valid that long),
// which bounds how far a fast GPU runs ahead to the depth of its ring -- the bounded channel.
}  // extern "C"

namespace {

struct SweepBoard {
    std::mutex mu;
    std::condition_variable cv;
    const rt_camera *cameras = nullptr;
    uint32_t n_frames = 0;
    uint32_t next_issue = 0;    // next frame of the list a worker may take
    uint32_t next_deliver = 0;  // frame the caller hands out next
    bool ready = false, abort = false;  // a worker offers frame `frame`; the caller gave up
    uint32_t frame = 0;
    const uint8_t *data = nullptr;
    size_t len = 0;
    int workers_left = 0;
    int rc = RT_OK;
    char err[512] = "";
};

struct BoardSource : FrameSource {
    SweepBoard &b;
    explicit BoardSource(SweepBoard &board) : b(board) {}
    int64_t next(rt_camera *cam, bool *use_cam) override {
        std::lock_guard<std::mutex> lock(b.mu);
        if (b.abort || b.next_issue >= b.n_frames) return -1;
        const uint32_t f = b.next_issue++;
        *use_cam = b.cameras != nullptr;
        if (b.cameras) *cam = b.cameras[f];
        return (int64_t)f;
    }
};

// a worker's frame callback: wait for the frame's turn, offer it, wait until the caller has consumed it
void board_offer(void *user, uint32_t frame, const uint8_t *data, size_t len) {
    SweepBoard &b = *static_cast<SweepBoard *>(user);
    std::unique_lock<std::mutex> lock(b.mu);
    b.cv.wait(lock, [&] { return b.abort || b.next_deliver == frame; });
    if (b.abort) return;  // let this GPU's pipeline run dry without hand-overs
    b.frame = frame;
    b.data = data;
    b.len = len;
    b.ready = true;
    b.cv.notify_all();
    b.cv.wait(lock, [&] { return b.abort || b.next_deliver != frame; });
}

static int sweep_multi_impl(rt_scene *const *scenes, int ngpu, const rt_camera *cameras, uint32_t n_frames, uint32_t width,
                            uint32_t height, uint32_t spp, OutKind kind, rt_frame_callback cb, void *user, rt_stats *stats,
                            const Animation *anim = nullptr) {
    if (!scenes || ngpu < 1) return fail(RT_ERR_INVALID, "need at least one scene");
    for (int g = 0; g < ngpu; g++) {
        int rc = check_frame_args(scenes[g], width, height, spp, 0, 1, height);
        if (rc != RT_OK) return rc;
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n_frames == 0) return RT_OK;
    if (ngpu == 1) {
        ListSource src(cameras, n_frames);
        return sweep_impl(scenes[0], src, width, height, spp, cb, user, stats, kind, anim);
    }
    RT_TRY(check_distinct_scenes(scenes, ngpu));  // each worker locks its own
    const double t0 = now_ms();
    const int variant = g_variant;  // the caller's choice travels to the workers (it is thread-local)
    SweepBoard board;
    board.cameras = cameras;
    board.n_frames = n_frames;
    board.workers_left = ngpu;
    std::vector<rt_stats> wstats((size_t)ngpu);
    std::vector<std::thread> workers;
    for (int g = 0; g < ngpu; g++) {
        memset(&wstats[(size_t)g], 0, sizeof(rt_stats));
        workers.emplace_back([&, g, variant]() {
            g_variant = variant;
            BoardSource src(board);
            const int rc = sweep_impl(scenes[g], src, width, height, spp, board_offer, &board, &wstats[(size_t)g], kind, anim);
            std::lock_guard<std::mutex> lock(board.mu);
            if (rc != RT_OK && board.rc == RT_OK) {
                board.rc = rc;
                snprintf(board.err, sizeof(board.err), "GPU %d: %.*s", scenes[g]->device, (int)sizeof(board.err) - 24, g_err);  // a long message is cut, never overrun
                board.abort = true;
            }
            board.workers_left--;
            board.cv.notify_all();
        });
    }
    {
        std::unique_lock<std::mutex> lock(board.mu);
        for (uint32_t f = 0; f < n_frames; f++) {
            board.cv.wait(lock, [&] { return board.abort || (board.ready && board.frame == f) || board.workers_left == 0; });
            if (!(board.ready && board.frame == f)) {  // a worker failed, or all ended without delivering frame f
                if (board.rc == RT_OK) {
                    board.rc = RT_ERR_CUDA;
                    snprintf(board.err, sizeof(board.err), "sweep workers ended before frame %u", f);
                }
                board.abort = true;
                board.cv.notify_all();
                break;
            }
            const uint8_t *data = board.data;
            const size_t len = board.len;
            lock.unlock();
            if (cb) cb(user, f, data, len);  // on the calling thread, without the board's lock
            lock.lock();
            board.ready = false;
            board.next_deliver = f + 1;
            board.cv.notify_all();
        }
    }
    for (std::thread &t : workers) t.join();
    if (board.rc != RT_OK) return fail(board.rc, "%s", board.err);
    if (stats) {
        stats->total_ms = now_ms() - t0;
        stats->primary_rays = (uint64_t)width * height * spp * spp * n_frames;
        for (const rt_stats &w : wstats) stats->kernel_launches += w.kernel_launches;
        stats->gpus = (uint32_t)ngpu;
        stats->variant_used = wstats[0].variant_used;
    }
    return RT_OK;
}

}  // namespace

extern "C" {

int rt_render_sweep_multi(rt_scene *const *scenes, int ngpu, const rt_camera *cameras, uint32_t n_frames, uint32_t width,
                          uint32_t height, uint32_t spp, int rgb, rt_frame_callback cb, void *user, rt_stats *stats) {
    return sweep_multi_impl(scenes, ngpu, cameras, n_frames, width, height, spp, rgb ? OutKind::RGB : OutKind::RGBA, cb,
                            user, stats);
}

int rt_render_sweep_png(rt_scene *const *scenes, int ngpu, const rt_camera *cameras, uint32_t n_frames, uint32_t width,
                        uint32_t height, uint32_t spp, rt_frame_callback cb, void *user, rt_stats *stats) {
    return sweep_multi_impl(scenes, ngpu, cameras, n_frames, width, height, spp, OutKind::PNG, cb, user, stats);
}

int rt_render_sweep_apng(rt_scene *const *scenes, int ngpu, const rt_camera *cameras, uint32_t n_frames, uint32_t width,
                         uint32_t height, uint32_t spp, uint16_t delay_num, uint16_t delay_den, rt_frame_callback cb,
                         void *user, rt_stats *stats) {
    size_t bound = 0;
    const int rc = rt_apng_bound(width, height, n_frames, &bound);
    if (rc != RT_OK) return rc;
    Animation anim;
    anim.n_frames = n_frames, anim.delay_num = delay_num, anim.delay_den = delay_den;
    return sweep_multi_impl(scenes, ngpu, cameras, n_frames, width, height, spp, OutKind::PNG, cb, user, stats, &anim);
}

uint64_t rt_atomic_fetch_add_u64(void *addr, uint64_t value) {
    return __atomic_fetch_add(static_cast<uint64_t *>(addr), value, __ATOMIC_SEQ_CST);
}

int rt_count_rays(const rt_scene *s, const rt_camera *camera, uint32_t width, uint32_t height, uint32_t spp,
                  uint32_t row_start, uint32_t row_stride, uint32_t row_count, uint64_t *primary, uint64_t *shadow) {
    if (!primary || !shadow) return fail(RT_ERR_INVALID, "NULL argument");
    uint64_t hits = 0;
    *primary = (uint64_t)width * row_count * spp * spp;
    *shadow = 0;
    return render_rows_impl(const_cast<rt_scene *>(s), camera, width, height, spp, row_start, row_stride, row_count,
                            nullptr, 0, nullptr, nullptr, nullptr, &hits, shadow);
}

int rt_trace_rays(const rt_scene *s, size_t n, const rt_ray *rays, rt_hit *hits) {
    if (!s || (n && (!rays || !hits))) return fail(RT_ERR_INVALID, "NULL argument");
    if (n == 0) return RT_OK;
    DeviceGuard guard(s->device);
    if (!guard.ok) return fail(RT_ERR_CUDA, "cannot select device %d", s->device);
    float *d_rays = nullptr, *d_hits = nullptr;
    CUDA_TRY(cudaMalloc(&d_rays, n * sizeof(rt_ray)));
    cudaError_t e = cudaMalloc(&d_hits, n * sizeof(rt_hit));
    if (e == cudaSuccess) e = cudaMemcpy(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = rt_launch_trace_rays(s->d_sph.as<float4>(), s->d_skip.as<uint32_t>(), s->n, n, d_rays, d_hits, nullptr);
    if (e == cudaSuccess) e = cudaMemcpy(hits, d_hits, n * sizeof(rt_hit), cudaMemcpyDeviceToHost);
    cudaFree(d_rays);
    if (d_hits) cudaFree(d_hits);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "trace_rays: %s", cudaGetErrorString(e));
    return RT_OK;
}

int rt_microbench_fp32(int device, int mode, double *tflops) {
    if (!tflops) return fail(RT_ERR_INVALID, "NULL argument");
    if (device < 0 || device >= rt_device_count()) return fail(RT_ERR_CUDA, "no CUDA device %d", device);
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    float *d_out = nullptr;
    CUDA_TRY(cudaMalloc(&d_out, 64));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int blocks = prop.multiProcessorCount * 8;
    const int iters = 20000;
    cudaError_t e = rt_launch_fp32_peak(mode, d_out, blocks, 2000, nullptr);  // warm-up / clock ramp
    if (e == cudaSuccess) e = cudaEventRecord(e0);
    if (e == cudaSuccess) e = rt_launch_fp32_peak(mode, d_out, blocks, iters, nullptr);
    if (e == cudaSuccess) e = cudaEventRecord(e1);
    if (e == cudaSuccess) e = cudaEventSynchronize(e1);
    float ms = 0.0f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d_out);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "fp32 microbench: %s", cudaGetErrorString(e));
    // 16 chains per thread; FFMA = 2 flop, FMUL+FADD pair = 2 flop in two instructions
    const double flop = (double)blocks * 256.0 * (double)iters * 16.0 * 2.0;
    *tflops = flop / (ms * 1e-3) / 1e12;
    return RT_OK;
}

int rt_selftest_math(uint32_t n, uint32_t seed, uint64_t mismatches[6]) {
    if (!mismatches) return fail(RT_ERR_INVALID, "NULL argument");
    if (rt_device_count() == 0) return fail(RT_ERR_CUDA, "no CUDA device");
    unsigned long long *d = nullptr;
    CUDA_TRY(cudaMalloc(&d, 48));
    cudaError_t e = cudaMemset(d, 0, 48);
    if (e == cudaSuccess) e = rt_launch_math_selftest(n, seed, d, nullptr);
    unsigned long long h[6] = {0, 0, 0, 0, 0, 0};
    if (e == cudaSuccess) e = cudaMemcpy(h, d, 48, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "math selftest: %s", cudaGetErrorString(e));
    for (int k = 0; k < 6; k++) mismatches[k] = h[k];
    return RT_OK;
}

int rt_measure_fp32_peak(int device, double *tflops, double *sm_clock_mhz) {
    int rc = rt_microbench_fp32(device, 0, tflops);
    if (rc != RT_OK) return rc;
    if (sm_clock_mhz) {
        cudaDeviceProp prop;
        DeviceGuard guard(device);
        CUDA_TRY(cudaGetDeviceProperties(&prop, device));
        // effective clock implied by the measured rate: 128 FFMA lanes per SM per cycle
        *sm_clock_mhz = *tflops * 1e12 / (2.0 * 128.0 * prop.multiProcessorCount) / 1e6;
    }
    return RT_OK;
}

// Diagnostic: candidate counts per cull tile of the most recent PHASED frame of this scene
// (walks the chunk chains on the host).  counts[2*t] = primary, counts[2*t+1] = shadow candidates;
// 0xffffffff = tile handled by the per-lane walk, 0xfffffffd (shadow only) = every shadow ray of the tile occluded
// by one leaf, no list.  Returns the number of tiles through *n_tiles.
int rt_debug_phased_tiles(const rt_scene *cs, uint32_t cap_tiles, uint32_t *n_tiles, uint32_t *counts) {
    rt_scene *s = const_cast<rt_scene *>(cs);
    if (!s || !n_tiles) return fail(RT_ERR_INVALID, "NULL argument");
    DeviceGuard guard(s->device);
    CUDA_TRY(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> lock(s->mu_scratch);
    auto it = std::find_if(s->scratch.begin(), s->scratch.end(), [](const auto &kv) { return kv.second.pool_count.ptr != nullptr; });
    if (it == s->scratch.end()) return fail(RT_ERR_INVALID, "no PHASED frame rendered yet");
    const StreamScratch &ph = it->second;
    const uint32_t nt = (uint32_t)(ph.hdr.cap / sizeof(uint4));
    *n_tiles = nt;
    if (!counts) return RT_OK;
    uint32_t used = 0;
    CUDA_TRY(cudaMemcpy(&used, ph.pool_count.ptr, sizeof(used), cudaMemcpyDeviceToHost));
    used = std::min(used, ph.pool_units);
    std::vector<uint4> hdr(nt), pool(used);
    CUDA_TRY(cudaMemcpy(hdr.data(), ph.hdr.ptr, (size_t)nt * sizeof(uint4), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(pool.data(), ph.pool.ptr, (size_t)used * sizeof(uint4), cudaMemcpyDeviceToHost));
    for (uint32_t t = 0; t < nt && t < cap_tiles; t++) {
        const uint32_t heads[2] = {hdr[t].x, hdr[t].y};
        for (int k = 0; k < 2; k++) {
            uint32_t n = 0, b = heads[k];
            if (b == 0xfffffffeu) n = 0xffffffffu;
            else if (b == 0xfffffffdu) n = 0xfffffffdu;  // COVERED: one leaf occludes every shadow ray of the tile
            else
                for (int guard_n = 0; b != 0xffffffffu && b < used && guard_n < 100000; guard_n++) n += pool[b].x, b = pool[b].y;
            counts[2 * t + k] = n;
        }
    }
    return RT_OK;
}

int rt_device_alloc(size_t bytes, void **out) {
    if (!out) return fail(RT_ERR_INVALID, "NULL argument");
    *out = nullptr;
    if (rt_device_count() == 0) return fail(RT_ERR_CUDA, "no CUDA device");
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 1);
    if (e != cudaSuccess) return fail(RT_ERR_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    return RT_OK;
}

void rt_device_free(void *p) {
    if (p) cudaFree(p);
}

int rt_ipc_export(const void *device_ptr, uint8_t handle[64]) {
    if (!device_ptr || !handle) return fail(RT_ERR_INVALID, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, const_cast<void *>(device_ptr)));
    memcpy(handle, &h, 64);
    return RT_OK;
}

int rt_ipc_open(const uint8_t handle[64], void **out) {
    if (!handle || !out) return fail(RT_ERR_INVALID, "NULL argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CUDA_TRY(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return RT_OK;
}

int rt_ipc_close(void *p) {
    if (!p) return RT_OK;
    CUDA_TRY(cudaIpcCloseMemHandle(p));
    return RT_OK;
}

int rt_memcpy(void *dst, const void *src, size_t bytes) {
    if (!dst || !src) return fail(RT_ERR_INVALID, "NULL argument");
    CUDA_TRY(cudaMemcpy(dst, src, bytes, cudaMemcpyDefault));
    return RT_OK;
}

int rt_memcpy2d_async(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width_bytes, size_t rows, void *stream) {
    if (!dst || !src) return fail(RT_ERR_INVALID, "NULL argument");
    if (width_bytes == 0 || rows == 0) return RT_OK;
    CUDA_TRY(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width_bytes, rows, cudaMemcpyDefault, (cudaStream_t)stream));
    return RT_OK;
}

int rt_pack_rgb_rows(const uint8_t *rgba_frame, uint8_t *rgb_frame, uint32_t width, uint32_t height, uint32_t row_start,
                     uint32_t row_stride, uint32_t row_block, void *stream) {
    if (!rgba_frame || !rgb_frame) return fail(RT_ERR_INVALID, "NULL argument");
    // height is also the grid's y extent at row_stride 1, whose limit is 65535
    if (width == 0 || height == 0 || width > 65535u || height > 65535u)
        return fail(RT_ERR_INVALID, "width/height must be in 1..65535 (got %u x %u)", width, height);
    int in_dev = -1, out_dev = -1, cur = -1;
    if (!is_device_ptr(rgba_frame, &in_dev) || !is_device_ptr(rgb_frame, &out_dev))
        return fail(RT_ERR_INVALID, "rgba_frame and rgb_frame must be device memory");
    CUDA_TRY(cudaGetDevice(&cur));
    if (in_dev != cur || out_dev != cur)
        return fail(RT_ERR_INVALID, "rgba_frame (device %d) and rgb_frame (device %d) must live on the current device %d", in_dev, out_dev, cur);
    if (row_block == 0 || row_stride < row_block) return fail(RT_ERR_INVALID, "row_stride %u is smaller than the row block %u", row_stride, row_block);
    if (((uint64_t)row_start * width) % 4 || ((uint64_t)row_stride * width) % 4)
        return fail(RT_ERR_INVALID, "row blocks must start at multiples of 4 pixels (row_start %u, row_stride %u, width %u)", row_start, row_stride, width);
    if ((((uintptr_t)rgba_frame) & 15) || (((uintptr_t)rgb_frame) & 3)) return fail(RT_ERR_INVALID, "buffers must be 16- / 4-byte aligned");
    CUDA_TRY(rt_launch_pack_rgb_blocks(rgba_frame, rgb_frame, width, height, row_start, row_stride, row_block, (cudaStream_t)stream));
    return RT_OK;
}

int rt_png_bound(uint32_t width, uint32_t height, size_t *bytes) {
    if (!bytes) return fail(RT_ERR_INVALID, "NULL argument");
    if (width == 0 || height == 0 || width > 65535u || height > 65535u)
        return fail(RT_ERR_INVALID, "width/height must be in 1..65535 (got %u x %u)", width, height);
    *bytes = rt_png_bound_bytes(width, height, nullptr);
    return RT_OK;
}

int rt_apng_bound(uint32_t width, uint32_t height, uint32_t n_frames, size_t *frame_bytes) {
    if (!frame_bytes) return fail(RT_ERR_INVALID, "NULL argument");
    size_t png = 0;
    const int rc = rt_png_bound(width, height, &png);
    if (rc != RT_OK) return rc;
    if (n_frames == 0) return fail(RT_ERR_INVALID, "an animation needs at least one frame");
    // the last chunk's sequence number, (n - 1)(C + 1) with C = bands + 2 chunks of zlib data per frame
    const uint64_t last_seq = (uint64_t)(n_frames - 1) * ((height + 15u) / 16u + 3u);
    if (last_seq > 0x7fffffffu)
        return fail(RT_ERR_INVALID, "%u frames of height %u need sequence numbers beyond 2^31 - 1", n_frames, height);
    const Animation anim{n_frames};
    *frame_bytes = rt_png_bound_bytes(width, height, &anim);
    return RT_OK;
}

// rt_encode_png (anim == nullptr) and rt_encode_apng_frame (frame `frame` of *anim)
static int encode_impl(const uint8_t *rgba, uint32_t width, uint32_t height, size_t pitch_bytes, uint8_t *file_out,
                       size_t cap, size_t *len_out, void *stream_, const Animation *anim, uint32_t frame) {
    if (!rgba || !len_out || (!file_out && cap)) return fail(RT_ERR_INVALID, "NULL argument");
    *len_out = 0;
    size_t bound = 0;
    int rc = anim ? rt_apng_bound(width, height, anim->n_frames, &bound) : rt_png_bound(width, height, &bound);
    if (rc != RT_OK) return rc;
    if (anim && frame >= anim->n_frames) return fail(RT_ERR_INVALID, "frame %u of an animation of %u frames", frame, anim->n_frames);
    const size_t row_bytes = (size_t)width * 4;
    if (pitch_bytes == 0) pitch_bytes = row_bytes;
    if (pitch_bytes < row_bytes) return fail(RT_ERR_INVALID, "pitch %zu is smaller than a row (%zu bytes)", pitch_bytes, row_bytes);
    int dev = -1, cur = -1;
    if (!is_device_ptr(rgba, &dev)) return fail(RT_ERR_INVALID, "rgba must be device memory");
    CUDA_TRY(cudaGetDevice(&cur));
    if (dev != cur) return fail(RT_ERR_INVALID, "rgba lives on device %d, the current device is %d", dev, cur);
    cudaStream_t stream = (cudaStream_t)stream_;
    // scratch per (device, stream), kept for the life of the process: no allocation per call once it has grown
    static std::mutex g_mu;
    // never deleted on purpose: no buffer is released in static destruction at process exit
    static auto *g_scratch = new std::map<std::pair<int, cudaStream_t>, PngEncodeScratch>();
    PngEncodeScratch *sc;
    {
        std::lock_guard<std::mutex> lock(g_mu);
        sc = &(*g_scratch)[std::make_pair(cur, stream)];
    }
    std::lock_guard<std::mutex> lock(sc->mu);
    unsigned long long len = 0;
    RT_TRY(queue_encode(rgba, pitch_bytes, width, height, anim, frame, bound, sc->scratch, sc->out, &len, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    if (len == 0 || len > bound) return fail(RT_ERR_CUDA, "PNG encoder returned %llu bytes (bound %zu)", len, bound);
    *len_out = (size_t)len;
    if (len > cap) return fail(RT_ERR_BUFFER, "%s holds %zu bytes, the %s needs %llu", anim ? "out" : "png_out", cap,
                               anim ? "frame" : "file", len);
    CUDA_TRY(cudaMemcpyAsync(file_out, sc->out.ptr, (size_t)len, cudaMemcpyDefault, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    return RT_OK;
}

int rt_encode_png(const uint8_t *rgba, uint32_t width, uint32_t height, size_t pitch_bytes, uint8_t *png_out, size_t cap,
                  size_t *len_out, void *stream) {
    return encode_impl(rgba, width, height, pitch_bytes, png_out, cap, len_out, stream, nullptr, 0);
}

int rt_encode_apng_frame(const uint8_t *rgba, uint32_t width, uint32_t height, size_t pitch_bytes, uint32_t frame,
                         uint32_t n_frames, uint16_t delay_num, uint16_t delay_den, uint8_t *out, size_t cap,
                         size_t *len_out, void *stream) {
    Animation anim;
    anim.n_frames = n_frames, anim.delay_num = delay_num, anim.delay_den = delay_den;
    return encode_impl(rgba, width, height, pitch_bytes, out, cap, len_out, stream, &anim, frame);
}

int rt_host_register(void *p, size_t bytes) {
    if (!p || !bytes) return fail(RT_ERR_INVALID, "NULL argument");
    if (rt_device_count() == 0) return fail(RT_ERR_CUDA, "no CUDA device");
    CUDA_TRY(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return RT_OK;
}

int rt_host_unregister(void *p) {
    if (!p) return RT_OK;
    CUDA_TRY(cudaHostUnregister(p));
    return RT_OK;
}

// Copy-only microbenchmark of the link the end-to-end numbers are bound by: `iters` device-to-host copies of
// `bytes` from the current device into pinned host memory, back to back on one stream, timed with CUDA events.
// The copies rotate over `n_buffers` host buffers (1..8): a sweep delivers frames into a ring of three, and a
// destination that is rewritten at once is a different load on the host than fresh memory.
int rt_microbench_d2h(size_t bytes, int iters, int n_buffers, double *gb_per_s) {
    if (!gb_per_s || bytes == 0 || iters < 1 || n_buffers < 1 || n_buffers > 8) return fail(RT_ERR_INVALID, "bad argument");
    if (rt_device_count() == 0) return fail(RT_ERR_CUDA, "no CUDA device");
    uint8_t *d = nullptr, *h[8] = {nullptr};
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    float ms = 0.0f;
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e == cudaSuccess) e = cudaMemset(d, 0x5a, bytes);
    for (int k = 0; k < n_buffers && e == cudaSuccess; k++) e = cudaHostAlloc((void **)&h[k], bytes, cudaHostAllocPortable);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    for (int i = 0; i < n_buffers && e == cudaSuccess; i++) e = cudaMemcpyAsync(h[i], d, bytes, cudaMemcpyDeviceToHost, st);  // warm-up
    if (e == cudaSuccess) e = cudaEventRecord(e0, st);
    for (int i = 0; i < iters && e == cudaSuccess; i++) e = cudaMemcpyAsync(h[i % n_buffers], d, bytes, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaEventRecord(e1, st);
    if (e == cudaSuccess) e = cudaEventSynchronize(e1);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (st) cudaStreamDestroy(st);
    for (int k = 0; k < n_buffers; k++)
        if (h[k]) cudaFreeHost(h[k]);
    if (d) cudaFree(d);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, "d2h microbench: %s", cudaGetErrorString(e));
    *gb_per_s = (double)bytes * iters / (ms * 1e-3) / 1e9;
    return RT_OK;
}

int rt_host_alloc(size_t bytes, void **out) {
    if (!out) return fail(RT_ERR_INVALID, "NULL argument");
    *out = nullptr;
    if (rt_device_count() == 0) return fail(RT_ERR_CUDA, "no CUDA device");
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) return fail(RT_ERR_NOMEM, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
    return RT_OK;
}

void rt_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

}  // extern "C"
