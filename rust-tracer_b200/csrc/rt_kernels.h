// rt_kernels.h -- host-side launch interface of rt_kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

enum { RT_KERNEL_LANE = 1, RT_KERNEL_WARP = 2, RT_KERNEL_TILE = 3, RT_KERNEL_PHASED = 4 };

// What a frame's kernels store per pixel: RGBA8 (4 bytes), or the four f32 values RGBA8 quantises (16 bytes, at
// out + row * pitch + x * 16).  Float output has LANE and PHASED kernels only, without diagnostics.
enum RtPixels { RT_PIXELS_RGBA8 = 0, RT_PIXELS_F32 = 1 };

namespace rt {
struct RenderParams;
}

// RT_PIXELS_F32 runs the LANE kernel whatever `variant` is.
cudaError_t rt_launch_render(int variant, bool diag, RtPixels fmt, const rt::RenderParams &p, cudaStream_t stream);
cudaError_t rt_launch_render_preview(const rt::RenderParams &p, cudaStream_t stream);
cudaError_t rt_launch_trace_rays(const float4 *sph, const uint32_t *skip, uint32_t n, size_t n_rays,
                                 const float *rays, float *hits, cudaStream_t stream);
cudaError_t rt_launch_pack_rgb(const uint8_t *rgba, uint8_t *rgb, size_t n_px, cudaStream_t stream);
cudaError_t rt_launch_pack_rgb_blocks(const uint8_t *rgba, uint8_t *rgb, uint32_t width, uint32_t height, uint32_t first,
                                      uint32_t stride, uint32_t block_rows, cudaStream_t stream);
cudaError_t rt_launch_fp32_peak(int mode, float *out, int blocks, int iters, cudaStream_t stream);

// TILE variant (rt_tile.cu): regular pyramids, 1 <= spp <= 4, orthonormal camera basis.
bool rt_tile_supported(const rt::RenderParams &p);
// PHASED variant: the same, 1 <= spp <= 8.
bool rt_phased_supported(const rt::RenderParams &p);
// shape 0: 16 ray slots per lane (largest tiles); shape 1: 4 slots per lane (4x more, shorter tiles)
cudaError_t rt_launch_render_tile(bool diag, const rt::RenderParams &p, cudaStream_t stream, int shape);
cudaError_t rt_launch_math_selftest(uint32_t n, uint32_t seed, unsigned long long *d_mismatch, cudaStream_t stream);

// PHASED variant (rt_phased.cu): the TILE algorithm as four launches on one stream.
void rt_phased_scratch(uint32_t width, uint32_t rows, uint32_t spp, int shape, size_t *winner_bytes, size_t *hdr_bytes,
                       uint32_t *pool_units);
cudaError_t rt_launch_render_phased(bool diag, RtPixels fmt, const rt::RenderParams &p, cudaStream_t stream, int shape);
