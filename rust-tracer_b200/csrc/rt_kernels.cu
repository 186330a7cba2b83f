// rt_kernels.cu -- sm_100a kernels for the rust-tracer hot path.
//
// One fused kernel per variant does, per pixel: ray generation (render.rs:238-243),
// primary closest-hit traversal (group.rs:72-83, primitive.rs:55-84), shading and
// the shadow ray (render.rs:188-214), spp^2 accumulation in the reference's sample
// order (render.rs:236-250) and RGBA8 quantisation (render.rs:92-109); the
// framebuffer is written exactly once.
//
// Variants (all bit-identical to the oracle by construction):
//   LANE  one thread per pixel; every lane walks the pre-order skip-pointer array
//         on its own (the direct stackless restatement of the recursion).
//   WARP  a warp owns an 8x4 pixel tile and walks the array ONCE for all 32 rays:
//         the node index is warp-uniform (one broadcast load per node), every lane
//         keeps the reference's own prune decision in a `resume` index (the lane
//         sleeps until the walk leaves the subtree it pruned), and a ballot
//         decides whether the walk descends or takes the skip link.
#include "rt_device.cuh"
#include "rt_kernels.h"

namespace rt {

static constexpr unsigned FULL = 0xffffffffu;
static constexpr int TILE_W = 8, TILE_H = 4;      // pixels per warp
static constexpr int WARPS_X = 4, WARPS_Y = 2;    // warps per block
static constexpr int BLOCK_THREADS = 32 * WARPS_X * WARPS_Y;

// ---------------------------------------------------------------------------
// WARP traversal: warp-uniform walk, per-lane reference prune state.
// ---------------------------------------------------------------------------
template <bool ANY>
RT_DEV void warp_traverse(const float4 *__restrict__ sph, const uint32_t *__restrict__ skip, uint32_t n, bool lane_on,
                          V3 o, V3 d, float &hitd, uint32_t &hit_idx) {
    if (!__any_sync(FULL, lane_on)) return;
    uint32_t resume = lane_on ? 0u : n;  // first node index at which this lane is awake again
    uint32_t i = 0;
    while (i < n) {
        float4 s = __ldg(&sph[i]);
        uint32_t sk = __ldg(&skip[i]);
        bool act = i >= resume;
        if (sk > i + 1) {  // group bound (warp-uniform branch)
            bool enter = false;
            if (act) {
                if (ANY)
                    enter = sphere_hit_any(s, o, d);
                else
                    enter = !(sphere_distance(s, o, d) >= hitd);
                if (!enter) resume = sk;  // this lane pruned the subtree (group.rs:73-75)
            }
            i = __any_sync(FULL, enter) ? i + 1 : sk;
        } else {  // leaf
            if (act) {
                if (ANY) {
                    if (sphere_hit_any(s, o, d)) {
                        hitd = 0.0f;
                        resume = n;  // any-hit: has_missed() is already false
                    }
                } else {
                    float dist = sphere_distance(s, o, d);
                    if (!(dist >= hitd)) {
                        hitd = dist;
                        hit_idx = i;
                    }
                }
            }
            i = i + 1;
            if (ANY) {
                if (!__any_sync(FULL, resume < n)) return;
            }
        }
    }
}

// ---------------------------------------------------------------------------
// The fused pixel kernel.  F32: the pixel is stored as the float4 {r, g, b, alpha} that RGBA8 output quantises.
// `tid` is threadIdx.x read in the __global__ function: there the compiler knows its range from the launch bounds,
// in a device function it does not, and the RGBA8 kernels would lose instructions that depend on it.
// ---------------------------------------------------------------------------
template <int VARIANT, bool DIAG, bool PREVIEW, bool F32>
__device__ __forceinline__ void render_body(const RenderParams &p, const uint32_t tid) {
    const int lane = tid & 31;
    const int warp = tid >> 5;
    const uint32_t lx = blockIdx.x * (TILE_W * WARPS_X) + (warp % WARPS_X) * TILE_W + (lane % TILE_W);
    const uint32_t j = blockIdx.y * (TILE_H * WARPS_Y) + (warp / WARPS_X) * TILE_H + (lane / TILE_W);
    const uint32_t cols = p.col_count ? p.col_count : p.width;  // column window (render_region buckets)
    const uint32_t step = PREVIEW ? p.px_step : 1u;             // preview: one traced pixel per step x step block
    const uint32_t x = (p.col_start + lx) * step;               // image column: what the ray is generated from
    const bool inside = lx < cols && j < p.row_count;
    if (VARIANT == RT_KERNEL_LANE && !inside) return;
    const uint32_t y = image_row(p, j) * step;

    const ShadeConsts K = shade_consts();
    const V3 eye = v3(p.eye[0], p.eye[1], p.eye[2]);
    const V3 light = v3(p.light[0], p.light[1], p.light[2]);
    const V3 to_light = vmulf(light, -1.0f);                  // render.rs:206
    const float sqrt_eps = fsqrt(1.1920928955078125e-07f);   // f32::EPSILON.sqrt(), render.rs:199

    V3 c = v3(0.0f, 0.0f, 0.0f);
    float alpha = 0.0f;
    unsigned n_hits = 0, n_shadow = 0;

    for (uint32_t ssx = 0; ssx < p.spp; ssx++) {
        for (uint32_t ssy = 0; ssy < p.spp; ssy++) {
            V3 d = primary_dir(p, x, y, ssx, ssy);
            float hitd = RT_INF;
            uint32_t hit_idx = 0;
            if (VARIANT == RT_KERNEL_LANE)
                lane_traverse<false>(p.sph, p.skip, p.n_nodes, eye, d, hitd, hit_idx);
            else
                warp_traverse<false>(p.sph, p.skip, p.n_nodes, inside, eye, d, hitd, hit_idx);

            uint8_t kind;
            bool want_shadow = false;
            float g = 0.0f;
            V3 sp = v3(0.0f, 0.0f, 0.0f);
            if (hitd == RT_INF) {  // render.rs:190-193
                c = vadd(c, K.background);
                kind = K_BACKGROUND;
            } else {
                n_hits++;
                V3 nrm = hit_normal(__ldg(&p.sph[hit_idx]), eye, d, hitd);
                g = vdot(nrm, light);  // render.rs:194
                if (g >= 0.0f) {       // render.rs:195-198
                    c = vadd(c, K.ambient);
                    kind = K_AWAY;
                } else {
                    // render.rs:199: (pos + dir*distance) + normal*(distance*sqrt(EPSILON))
                    sp = vadd(vadd(eye, vmulf(d, hitd)), vmulf(nrm, fmul(hitd, sqrt_eps)));
                    want_shadow = true;
                    kind = K_LIT;
                }
            }
            float sh = RT_INF;
            uint32_t dummy = 0;
            if (VARIANT == RT_KERNEL_LANE) {
                if (want_shadow) lane_traverse<true>(p.sph, p.skip, p.n_nodes, sp, to_light, sh, dummy);
            } else {
                warp_traverse<true>(p.sph, p.skip, p.n_nodes, want_shadow && inside, sp, to_light, sh, dummy);
            }
            if (want_shadow) {
                n_shadow++;
                float ng = -g;
                if (sh == RT_INF) {  // render.rs:208-210
                    c = vadd(vadd(c, vmulf(K.object, ng)), K.ambient);
                    alpha = fadd(alpha, 1.0f);
                } else {  // render.rs:211-214
                    c = vadd(vadd(c, K.background), vmulf(K.ambient, ng));
                    kind = K_SHADOWED;
                }
            }
            if (DIAG && p.kinds && inside)
                p.kinds[((size_t)j * cols + lx) * (p.spp * p.spp) + ssx * p.spp + ssy] = kind;
        }
    }

    if (inside) {
        float recip = frecip(fmul((float)p.spp, (float)p.spp));  // render.rs:219-220
        c = vmulf(c, recip);
        alpha = fmul(alpha, recip);
        if constexpr (F32) {
            *reinterpret_cast<float4 *>(p.out + (size_t)out_row(p, j) * p.pitch + (size_t)lx * 16) = make_float4(c.x, c.y, c.z, alpha);
            return;
        }
        uint32_t px = scale_u8(c.x) | (scale_u8(c.y) << 8) | (scale_u8(c.z) << 16) | (scale_u8(alpha) << 24);
        if (PREVIEW) {  // the block's pixels that lie inside the image, each row of the block contiguous
            const uint32_t x1 = min(x + step, p.width), y1 = min(y + step, p.height);
            for (uint32_t yy = y; yy < y1; yy++) {
                uint32_t *row = reinterpret_cast<uint32_t *>(p.out + (size_t)yy * p.pitch);
                for (uint32_t xx = x; xx < x1; xx++) row[xx] = px;
            }
        } else {
            *reinterpret_cast<uint32_t *>(p.out + (size_t)out_row(p, j) * p.pitch + (size_t)lx * 4) = px;
        }
    }
    if (DIAG && p.ray_counters) {
        if (!inside) {
            n_hits = 0;
            n_shadow = 0;
        }
        if (VARIANT == RT_KERNEL_LANE) {
            atomicAdd(&p.ray_counters[0], (unsigned long long)n_hits);
            atomicAdd(&p.ray_counters[1], (unsigned long long)n_shadow);
        } else {
            n_hits = __reduce_add_sync(FULL, n_hits);
            n_shadow = __reduce_add_sync(FULL, n_shadow);
            if (lane == 0) {
                atomicAdd(&p.ray_counters[0], (unsigned long long)n_hits);
                atomicAdd(&p.ray_counters[1], (unsigned long long)n_shadow);
            }
        }
    }
}

template <int VARIANT, bool DIAG, bool PREVIEW = false>
__global__ void __launch_bounds__(BLOCK_THREADS) render_kernel(const RenderParams p) {
    render_body<VARIANT, DIAG, PREVIEW, false>(p, threadIdx.x);
}

// LANE with float output: the fallback of float frames outside PHASED's domain.
__global__ void __launch_bounds__(BLOCK_THREADS) render_lane_f32_kernel(const RenderParams p) {
    render_body<RT_KERNEL_LANE, false, false, true>(p, threadIdx.x);
}

// Closest-hit traversal of arbitrary rays (rt_trace_rays): group.rs:72-83 from Hit::missed().
__global__ void trace_rays_kernel(const float4 *__restrict__ sph, const uint32_t *__restrict__ skip, uint32_t n,
                                  size_t n_rays, const float *__restrict__ rays, float *__restrict__ hits) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rays) return;
    V3 o = v3(rays[i * 6 + 0], rays[i * 6 + 1], rays[i * 6 + 2]);
    V3 d = v3(rays[i * 6 + 3], rays[i * 6 + 4], rays[i * 6 + 5]);
    float hitd = RT_INF;
    uint32_t idx = 0;
    lane_traverse<false>(sph, skip, n, o, d, hitd, idx);
    V3 nrm = v3(0.0f, 0.0f, 0.0f);
    if (hitd != RT_INF) nrm = hit_normal(__ldg(&sph[idx]), o, d, hitd);
    hits[i * 4 + 0] = hitd;
    hits[i * 4 + 1] = nrm.x;
    hits[i * 4 + 2] = nrm.y;
    hits[i * 4 + 3] = nrm.z;
}

// RGBA8 -> RGB8 (the PPM sink drops alpha, render.rs:389-397): 4 pixels per thread, 16 bytes in, 12 out.
__global__ void pack_rgb_kernel(const uint32_t *__restrict__ rgba, uint32_t *__restrict__ rgb, size_t n_quads,
                                size_t n_px) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < n_quads) {
        const uint4 v = reinterpret_cast<const uint4 *>(rgba)[q];
        const uint32_t a = v.x & 0xffffffu, b = v.y & 0xffffffu, c = v.z & 0xffffffu, d = v.w & 0xffffffu;
        rgb[3 * q + 0] = a | (b << 24);
        rgb[3 * q + 1] = (b >> 8) | (c << 16);
        rgb[3 * q + 2] = (c >> 16) | (d << 8);
    }
    if (q == 0) {  // up to 3 trailing pixels
        uint8_t *o = reinterpret_cast<uint8_t *>(rgb);
        const uint8_t *i = reinterpret_cast<const uint8_t *>(rgba);
        for (size_t px = n_quads * 4; px < n_px; px++)
            for (int k = 0; k < 3; k++) o[px * 3 + k] = i[px * 4 + k];
    }
}

// The same for the row blocks one GPU owns of a frame-shaped buffer: blocks of `block_rows` rows starting at row
// first + k * stride (k = blockIdx.y), packed to the same rows of a frame-shaped RGB8 buffer.  Block starts are
// multiples of 4 pixels (the host checks it), so quads never straddle a block.
__global__ void pack_rgb_blocks_kernel(const uint8_t *__restrict__ rgba, uint8_t *__restrict__ rgb, uint32_t width,
                                       uint32_t height, uint32_t first, uint32_t stride, uint32_t block_rows) {
    const uint32_t row0 = first + blockIdx.y * stride;
    if (row0 >= height) return;
    const uint32_t rows = min(block_rows, height - row0);
    const size_t px0 = (size_t)row0 * width, n_px = (size_t)rows * width, n_quads = n_px / 4;
    const uint4 *src = reinterpret_cast<const uint4 *>(rgba + px0 * 4);
    uint32_t *dst = reinterpret_cast<uint32_t *>(rgb + px0 * 3);
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_quads; q += (size_t)gridDim.x * blockDim.x) {
        const uint4 v = src[q];
        const uint32_t a = v.x & 0xffffffu, b = v.y & 0xffffffu, c = v.z & 0xffffffu, d = v.w & 0xffffffu;
        dst[3 * q + 0] = a | (b << 24);
        dst[3 * q + 1] = (b >> 8) | (c << 16);
        dst[3 * q + 2] = (c >> 16) | (d << 8);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)  // up to 3 trailing pixels of the block
        for (size_t px = n_quads * 4; px < n_px; px++)
            for (int k = 0; k < 3; k++) rgb[(px0 + px) * 3 + k] = rgba[(px0 + px) * 4 + k];
}

// Register-resident FP32 chains: the live roofline denominator.
// mode 0: FFMA; mode 1: alternating FMUL / FADD (the unfused mix the parity rule forces);
// mode 2: packed FFMA2 (sm_100 f32x2); mode 3: packed FMUL2 / FADD2.
template <int MODE>
__global__ void __launch_bounds__(256) fp32_peak_kernel(float *out, int iters, float a, float b) {
    float s = 0.0f;
    if (MODE < 2) {
        float r[16];
#pragma unroll
        for (int k = 0; k < 16; k++) r[k] = (float)(threadIdx.x + k) * 1e-3f;
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 16; k++) {
                if (MODE == 0) {
                    r[k] = __fmaf_rn(r[k], a, b);
                } else {
                    r[k] = __fmul_rn(r[k], a);
                    r[k] = __fadd_rn(r[k], b);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 16; k++) s += r[k];
    } else {
        float2 r[8];
        const float2 a2 = make_float2(a, a), b2 = make_float2(b, b);
#pragma unroll
        for (int k = 0; k < 8; k++) r[k] = make_float2((float)(threadIdx.x + k) * 1e-3f, (float)(threadIdx.x + k) * 2e-3f);
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                if (MODE == 2) {
                    r[k] = __ffma2_rn(r[k], a2, b2);
                } else {
                    r[k] = __fmul2_rn(r[k], a2);
                    r[k] = __fadd2_rn(r[k], b2);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 8; k++) s += r[k].x + r[k].y;
    }
    if (s == 12345.678f) out[0] = s;  // keep the chains alive
}

}  // namespace rt

// ---------------------------------------------------------------------------
// Host-side launchers (called from rt_api.cpp through rt_kernels.h).
// ---------------------------------------------------------------------------
using namespace rt;

cudaError_t rt_launch_render(int variant, bool diag, RtPixels fmt, const RenderParams &p, cudaStream_t stream) {
    dim3 block(BLOCK_THREADS);
    const uint32_t cols = p.col_count ? p.col_count : p.width;
    dim3 grid((cols + TILE_W * WARPS_X - 1) / (TILE_W * WARPS_X),
              (p.row_count + TILE_H * WARPS_Y - 1) / (TILE_H * WARPS_Y));
    if (grid.x == 0 || grid.y == 0) return cudaSuccess;
    if (fmt == RT_PIXELS_F32) {
        render_lane_f32_kernel<<<grid, block, 0, stream>>>(p);
    } else if (variant == RT_KERNEL_LANE) {
        if (diag)
            render_kernel<RT_KERNEL_LANE, true><<<grid, block, 0, stream>>>(p);
        else
            render_kernel<RT_KERNEL_LANE, false><<<grid, block, 0, stream>>>(p);
    } else {
        if (diag)
            render_kernel<RT_KERNEL_WARP, true><<<grid, block, 0, stream>>>(p);
        else
            render_kernel<RT_KERNEL_WARP, false><<<grid, block, 0, stream>>>(p);
    }
    return cudaGetLastError();
}

// One ray per px_step x px_step block (p.col_count x p.row_count blocks), colour replicated over the block.
cudaError_t rt_launch_render_preview(const RenderParams &p, cudaStream_t stream) {
    dim3 block(BLOCK_THREADS);
    dim3 grid((p.col_count + TILE_W * WARPS_X - 1) / (TILE_W * WARPS_X),
              (p.row_count + TILE_H * WARPS_Y - 1) / (TILE_H * WARPS_Y));
    if (grid.x == 0 || grid.y == 0 || p.px_step == 0) return cudaSuccess;
    render_kernel<RT_KERNEL_LANE, false, true><<<grid, block, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t rt_launch_trace_rays(const float4 *sph, const uint32_t *skip, uint32_t n, size_t n_rays,
                                 const float *rays, float *hits, cudaStream_t stream) {
    if (n_rays == 0) return cudaSuccess;
    unsigned blocks = (unsigned)((n_rays + 127) / 128);
    trace_rays_kernel<<<blocks, 128, 0, stream>>>(sph, skip, n, n_rays, rays, hits);
    return cudaGetLastError();
}

cudaError_t rt_launch_pack_rgb(const uint8_t *rgba, uint8_t *rgb, size_t n_px, cudaStream_t stream) {
    if (n_px == 0) return cudaSuccess;
    const size_t quads = n_px / 4;
    const unsigned blocks = (unsigned)((quads + 255) / 256);
    pack_rgb_kernel<<<blocks ? blocks : 1, 256, 0, stream>>>(reinterpret_cast<const uint32_t *>(rgba),
                                                              reinterpret_cast<uint32_t *>(rgb), quads, n_px);
    return cudaGetLastError();
}

cudaError_t rt_launch_pack_rgb_blocks(const uint8_t *rgba, uint8_t *rgb, uint32_t width, uint32_t height, uint32_t first,
                                      uint32_t stride, uint32_t block_rows, cudaStream_t stream) {
    if (first >= height || width == 0 || block_rows == 0) return cudaSuccess;
    const uint32_t n_blocks = (height - first + stride - 1) / stride;
    const size_t quads = (size_t)block_rows * width / 4;
    unsigned gx = (unsigned)((quads + 255) / 256);
    if (gx > 1024) gx = 1024;
    pack_rgb_blocks_kernel<<<dim3(gx ? gx : 1, n_blocks), 256, 0, stream>>>(rgba, rgb, width, height, first, stride, block_rows);
    return cudaGetLastError();
}

cudaError_t rt_launch_fp32_peak(int mode, float *out, int blocks, int iters, cudaStream_t stream) {
    if (mode == 0)
        fp32_peak_kernel<0><<<blocks, 256, 0, stream>>>(out, iters, 1.0000001f, 1e-7f);
    else if (mode == 1)
        fp32_peak_kernel<1><<<blocks, 256, 0, stream>>>(out, iters, 1.0000001f, 1e-7f);
    else if (mode == 2)
        fp32_peak_kernel<2><<<blocks, 256, 0, stream>>>(out, iters, 1.0000001f, 1e-7f);
    else
        fp32_peak_kernel<3><<<blocks, 256, 0, stream>>>(out, iters, 1.0000001f, 1e-7f);
    return cudaGetLastError();
}
