// rt_exr.h -- host-side launch interface of rt_exr.cu (OpenEXR files encoded on the device).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

// Worst-case file size of a width x height frame, with (aov) or without the AOV channels: the header, the offset
// table, and every chunk stored raw (8 + its uncompressed bytes), which is the size of a file whose chunks all fall
// back to raw.
size_t rt_exr_bound_bytes(uint32_t width, uint32_t height, bool aov);
// Device scratch one encode needs (piece staging and per-piece records).
size_t rt_exr_scratch_bytes(uint32_t width, uint32_t height, bool aov);
// Encode the float colour frame `rgba` (device, {r, g, b, alpha} per pixel, `rgba_pitch` bytes per row) and, when
// `aov` is not null, the AOV frame `aov` (device, 8 floats per pixel, `aov_pitch` bytes per row) into `out` (device,
// >= rt_exr_bound_bytes) and store its length in *len_word (device), asynchronously on `stream`.  `scratch` holds
// rt_exr_scratch_bytes; one encode at a time may use it.
cudaError_t rt_launch_exr_encode(const float *rgba, size_t rgba_pitch, const float *aov, size_t aov_pitch,
                                 uint32_t width, uint32_t height, void *scratch, uint8_t *out,
                                 unsigned long long *len_word, cudaStream_t stream);
