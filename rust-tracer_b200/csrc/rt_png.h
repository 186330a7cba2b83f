// rt_png.h -- host-side launch interface of rt_png.cu (PNG files encoded on the device).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

// The animated PNG a frame belongs to: its frame count and how long each frame shows (delay_num / delay_den s).
// Where an entry point takes `const Animation *`, nullptr means a stand-alone PNG file.
struct Animation {
    uint32_t n_frames = 0;
    uint16_t delay_num = 0, delay_den = 0;
};

// Worst-case file size of a width x height frame (every raw-row byte at most 9 bits, plus all framing); with `anim`,
// the worst-case payload of one of its frames: that bound, acTL, fcTL and every chunk's sequence number.
size_t rt_png_bound_bytes(uint32_t width, uint32_t height, const Animation *anim);
// Device scratch one encode needs (row staging, run masks, per-row and per-band records).
size_t rt_png_scratch_bytes(uint32_t width, uint32_t height);
// Encode the RGBA8 frame `rgba` (device, `pitch` bytes per row) into `out` (device, >= rt_png_bound_bytes) and
// store its length in *len_word (device), asynchronously on `stream`.  `scratch` holds rt_png_scratch_bytes; one
// encode at a time may use it.  Without `anim`, `out` gets the PNG file; with it, frame `frame` (< n_frames) of that
// animation: the frame's payload, where the payloads of frames 0 .. n_frames-1 back to back are the file.
cudaError_t rt_launch_png_encode(const uint8_t *rgba, size_t pitch, uint32_t width, uint32_t height, const Animation *anim,
                                 uint32_t frame, void *scratch, uint8_t *out, unsigned long long *len_word,
                                 cudaStream_t stream);
