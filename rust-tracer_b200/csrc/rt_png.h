// rt_png.h -- host-side launch interface of rt_png.cu (PNG files encoded on the device).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

// Worst-case file size of a width x height frame (every raw-row byte at most 9 bits, plus all framing).
size_t rt_png_bound_bytes(uint32_t width, uint32_t height);
// Worst-case payload of one APNG frame (rt_launch_apng_encode): the PNG bound, acTL, fcTL and every chunk's sequence
// number.
size_t rt_apng_bound_bytes(uint32_t width, uint32_t height);
// Device scratch one encode needs (row staging, run masks, per-row and per-band records).
size_t rt_png_scratch_bytes(uint32_t width, uint32_t height);
// Encode the RGBA8 frame `rgba` (device, `pitch` bytes per row) into `out` (device, >= rt_png_bound_bytes) and
// store the file length in *len_word (device), asynchronously on `stream`.  `scratch` holds
// rt_png_scratch_bytes; one encode at a time may use it.
cudaError_t rt_launch_png_encode(const uint8_t *rgba, size_t pitch, uint32_t width, uint32_t height, void *scratch,
                                 uint8_t *out, unsigned long long *len_word, cudaStream_t stream);
// The same encode, written as frame `frame` (< n_frames) of an animated PNG whose frames each show for
// delay_num / delay_den seconds: the frame's payload goes to `out` (device, >= rt_apng_bound_bytes) and its length
// to *len_word.  The payloads of frames 0 .. n_frames-1 back to back are the file.
cudaError_t rt_launch_apng_encode(const uint8_t *rgba, size_t pitch, uint32_t width, uint32_t height, uint32_t frame,
                                  uint32_t n_frames, uint16_t delay_num, uint16_t delay_den, void *scratch, uint8_t *out,
                                  unsigned long long *len_word, cudaStream_t stream);
