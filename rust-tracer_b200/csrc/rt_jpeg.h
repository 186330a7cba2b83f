// rt_jpeg.h -- host-side launch interface of rt_jpeg.cu (JPEG files encoded on the device).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

// Worst-case file size of a width x height frame at any quality: the header, every MCU row at its worst (each
// block at the most bits a block can code to, a padding byte, all of it doubled for 0xFF stuffing, its RST
// marker), and EOI.
size_t rt_jpeg_bound_bytes(uint32_t width, uint32_t height);
// Device scratch one encode needs (coefficients, per-block bit lengths and offsets, row staging, per-row records).
size_t rt_jpeg_scratch_bytes(uint32_t width, uint32_t height);
// Encode the RGBA8 frame `rgba` (device, `pitch` bytes per row; alpha is dropped) at `quality` (1..100) into `out`
// (device, >= rt_jpeg_bound_bytes) and store its length in *len_word (device), asynchronously on `stream`.
// `scratch` holds rt_jpeg_scratch_bytes; one encode at a time may use it.
cudaError_t rt_launch_jpeg_encode(const uint8_t *rgba, size_t pitch, uint32_t width, uint32_t height, int quality,
                                  void *scratch, uint8_t *out, unsigned long long *len_word, cudaStream_t stream);
