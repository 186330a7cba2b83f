// render.hpp -- host-side mirror of the reference crate's public interface
// (src/rust/lib.rs:8: Scene, Renderer, RenderOptions, PPMStdoutRGBABufferWriter,
// FileOrAnyWriter) over the C ABI of librtrace_b200.so.
//
// The names, argument meaning and error behaviour follow src/rust/render.rs; what
// changed is the engine underneath Renderer::render: the thread pool + bounded
// channel of 64x64 buckets (render.rs:271-307) became kernel launches per GPU over
// interleaved row blocks that every GPU copies straight into the host frame.  The writer trait is kept as the seam
// for output sinks (render.rs:20-30).
#pragma once
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <memory>
#include <unistd.h>
#include <stdexcept>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "rtrace.h"

namespace sphere_tracer {

// A failed `assert!`/`unwrap()` in the reference is a panic (exit code 101).
struct Panic : std::runtime_error {
    explicit Panic(const std::string &m) : std::runtime_error(m) {}
};

inline void rt_check(int rc, const char *what) {
    if (rc != RT_OK) throw Panic(std::string(what) + ": " + rt_last_error());
}

// render.rs:33-38
struct RenderOptions {
    uint16_t width = 1024;
    uint16_t height = 1024;
    uint16_t samples_per_pixel = 1;
};

// render.rs:42-72 (t > b; b is the upper image row)
struct ImageRegion {
    uint16_t l = 0, t = 0, r = 0, b = 0;
    uint16_t width() const { return r - l; }
    uint16_t height() const { return t - b; }
    size_t area() const { return (size_t)width() * height(); }
    bool contains(const ImageRegion &o) const { return o.l >= l && o.b >= b && o.t <= t && o.r <= r; }
    size_t buffer_offset(uint16_t x, uint16_t y) const { return (size_t)(y - b) * width() + (size_t)(x - l); }
    bool operator==(const ImageRegion &o) const { return l == o.l && t == o.t && r == o.r && b == o.b; }
};

// render.rs:74-135.  Pixels live in pinned host memory so the device-to-host copy
// of a frame runs at PCIe rate.
class RGBABuffer {
  public:
    explicit RGBABuffer(const ImageRegion &r) : reg_(r), len_(r.area() * components()) {
        void *p = nullptr;
        rt_check(rt_host_alloc(len_, &p), "RGBABuffer::new");
        buf_ = static_cast<uint8_t *>(p);
    }
    ~RGBABuffer() { rt_host_free(buf_); }
    RGBABuffer(const RGBABuffer &) = delete;
    RGBABuffer &operator=(const RGBABuffer &) = delete;
    static size_t components() { return 4; }
    uint8_t *data() { return buf_; }
    const uint8_t *buffer() const { return buf_; }
    // Fill from a finished frame of the same region (the sweep hands out library-owned pinned memory).
    void copy_from(const uint8_t *rgba, size_t len) { memcpy(buf_, rgba, len < len_ ? len : len_); }
    size_t len() const { return len_; }
    const ImageRegion &region() const { return reg_; }

    // render.rs:112-126
    void set_pixels_from_buffer(const RGBABuffer &b) {
        if (!reg_.contains(b.reg_)) throw Panic("assertion failed: self.reg.contains(&b.reg)");
        if (reg_ == b.reg_) {
            memcpy(buf_, b.buf_, len_);
            return;
        }
        size_t w = (size_t)b.reg_.width() * components();
        for (uint16_t y = b.reg_.b; y < b.reg_.t; y++) {
            size_t bl = reg_.buffer_offset(b.reg_.l, y) * components();
            size_t their_bl = b.reg_.buffer_offset(b.reg_.l, y) * components();
            memcpy(buf_ + bl, b.buf_ + their_bl, w);
        }
    }

  private:
    ImageRegion reg_;
    size_t len_;
    uint8_t *buf_ = nullptr;
};

// render.rs:20-30
struct RGBABufferWriter {
    virtual ~RGBABufferWriter() {}
    virtual void begin(uint16_t x, uint16_t y) = 0;
    virtual void write_rgba_buffer(const RGBABuffer &buffer) = 0;
};

// render.rs:313-316
struct FileOrAnyWriter {
    FILE *f = nullptr;
    bool is_file = false;
    static FileOrAnyWriter any_writer_stdout() { return FileOrAnyWriter{stdout, false}; }
    static FileOrAnyWriter file_writer(FILE *fp) { return FileOrAnyWriter{fp, true}; }
};

// render.rs:319-434: P6 (rgb) or P5 (grey) with the alpha channel stripped; the
// whole image is (re)written from the top each time; final write on destruction.
// The progressive rewrite follows render.rs:427-432: a buffer arriving at a file sink
// triggers a rewrite of the whole file when none happened yet or the last one is at
// least a second old.  With a GPU frame arriving in one buffer that is one write per
// frame; a caller feeding bands (one per GPU) gets the reference's behaviour.
class PPMStdoutRGBABufferWriter : public RGBABufferWriter {
  public:
    PPMStdoutRGBABufferWriter(bool write_rgb, FileOrAnyWriter *writer) : out_(writer), rgb_(write_rgb) {}
    ~PPMStdoutRGBABufferWriter() override {
        try {
            write_buffer_with_header();
        } catch (...) {
        }
    }
    void begin(uint16_t x, uint16_t y) override {
        width_ = x;
        height_ = y;
        have_dims_ = true;
        ImageRegion r;
        r.l = 0, r.r = x, r.b = 0, r.t = y;
        image_.reset(new RGBABuffer(r));
    }
    void write_rgba_buffer(const RGBABuffer &buffer) override {
        if (!image_) throw Panic("called `Option::unwrap()` on a `None` value");
        image_->set_pixels_from_buffer(buffer);
        dirty_ = true;
        // "Flush full image right away" (render.rs:426-432): at most once per second
        const auto now = std::chrono::steady_clock::now();
        if (out_->is_file && (!written_once_ || last_written_at_ + std::chrono::seconds(1) <= now)) {
            written_once_ = true;
            last_written_at_ = now;
            write_buffer_with_header();
        }
    }

  private:
    void write_buffer_with_header() {
        if (!dirty_) return;
        FILE *f = out_->f;
        if (out_->is_file) {
            fflush(f);
            if (ftruncate(fileno(f), 0) != 0) throw Panic("set_len(0) failed");
            rewind(f);
        }
        if (!have_dims_) throw Panic("begin() called");
        fprintf(f, "%s\n%u %u\n255\n", rgb_ ? "P6" : "P5", (unsigned)width_, (unsigned)height_);
        const uint8_t *buf = image_->buffer();
        const size_t n = image_->len() / 4;
        std::vector<uint8_t> line;
        line.resize(n * (rgb_ ? 3 : 1));
        for (size_t i = 0; i < n; i++) {
            const uint8_t *b = buf + i * 4;
            if (rgb_) {
                line[i * 3 + 0] = b[0];
                line[i * 3 + 1] = b[1];
                line[i * 3 + 2] = b[2];
            } else {
                line[i] = (uint8_t)(((float)b[0] + (float)b[1] + (float)b[2]) / 3.0f);  // render.rs:399
            }
        }
        if (fwrite(line.data(), 1, line.size(), f) != line.size()) throw Panic("write_all failed");
        fflush(f);
        dirty_ = false;
    }
    FileOrAnyWriter *out_;
    uint16_t width_ = 0, height_ = 0;
    bool have_dims_ = false;
    std::unique_ptr<RGBABuffer> image_;
    bool rgb_;
    bool dirty_ = false;
    bool written_once_ = false;  // last_written_at: Option<Instant> (render.rs:325)
    std::chrono::steady_clock::time_point last_written_at_;
};

// Extension (SURVEY 8f N3): a sink that writes what the `.tga` extension promises.  Layout as the
// reference's Go sibling writes it (src/go/gotrace.go:248-280): 18-byte header, image type 2
// (uncompressed true colour), 24 bits per pixel, BGR, rows bottom-up.  Same seam, same buffering
// rules as the PPM sink; selected with `--format tga` (the default stays the reference's P6).
inline void write_tga(FILE *f, uint16_t width, uint16_t height, const uint8_t *px, size_t stride, size_t comps) {
    uint8_t header[18] = {0};
    header[2] = 2;
    header[12] = (uint8_t)(width & 0xff), header[13] = (uint8_t)(width >> 8);
    header[14] = (uint8_t)(height & 0xff), header[15] = (uint8_t)(height >> 8);
    header[16] = 24;
    if (fwrite(header, 1, sizeof(header), f) != sizeof(header)) throw Panic("write_all failed");
    std::vector<uint8_t> line((size_t)width * 3);
    for (uint32_t y = height; y-- > 0;) {  // bottom row first
        const uint8_t *row = px + (size_t)y * stride;
        for (uint32_t x = 0; x < width; x++) {
            line[x * 3 + 0] = row[x * comps + 2];
            line[x * 3 + 1] = row[x * comps + 1];
            line[x * 3 + 2] = row[x * comps + 0];
        }
        if (fwrite(line.data(), 1, line.size(), f) != line.size()) throw Panic("write_all failed");
    }
    fflush(f);
}

// Extension: a colour PFM of a frame's pixels before quantisation -- "PF", the size, scale -1.0 (little-endian
// samples), then the rows from the bottom up as 32-bit float RGB.  `px` holds `height` rows of {r, g, b, alpha}
// floats, `stride` floats apart; alpha is dropped, as the P6 sink drops it.
inline void write_pfm(FILE *f, uint16_t width, uint16_t height, const float *px, size_t stride) {
    fprintf(f, "PF\n%u %u\n-1.0\n", (unsigned)width, (unsigned)height);
    std::vector<uint8_t> line((size_t)width * 12);
    for (uint32_t y = height; y-- > 0;) {  // bottom row first
        const float *row = px + (size_t)y * stride;
        for (uint32_t x = 0; x < width; x++)
            for (int c = 0; c < 3; c++) {
                uint32_t bits;
                memcpy(&bits, &row[x * 4 + c], 4);
                for (int b = 0; b < 4; b++) line[(x * 3 + c) * 4 + b] = (uint8_t)(bits >> (8 * b));
            }
        if (fwrite(line.data(), 1, line.size(), f) != line.size()) throw Panic("write_all failed");
    }
    fflush(f);
}

class TGARGBABufferWriter : public RGBABufferWriter {
  public:
    explicit TGARGBABufferWriter(FileOrAnyWriter *writer) : out_(writer) {}
    ~TGARGBABufferWriter() override {
        try {
            flush();
        } catch (...) {
        }
    }
    void begin(uint16_t x, uint16_t y) override {
        width_ = x, height_ = y;
        ImageRegion r;
        r.l = 0, r.r = x, r.b = 0, r.t = y;
        image_.reset(new RGBABuffer(r));
    }
    void write_rgba_buffer(const RGBABuffer &buffer) override {
        if (!image_) throw Panic("called `Option::unwrap()` on a `None` value");
        image_->set_pixels_from_buffer(buffer);
        dirty_ = true;
    }

  private:
    void flush() {
        if (!dirty_) return;
        write_tga(out_->f, width_, height_, image_->buffer(), (size_t)width_ * 4, 4);
        dirty_ = false;
    }
    FileOrAnyWriter *out_;
    uint16_t width_ = 0, height_ = 0;
    std::unique_ptr<RGBABuffer> image_;
    bool dirty_ = false;
};

// render.rs:138-167: one replica of the flattened scene per GPU.
class Scene {
  public:
    // Scene::default() generalised by `level`; replicated on devices 0..gpus-1.  The replicas are created
    // concurrently, one host thread per GPU: creating a CUDA context takes about a second per device, and
    // one after the other that was 7-8 s of start-up on an 8-GPU box.
    explicit Scene(uint32_t level = 8, int gpus = 1) {
        const int n = gpus < 1 ? 1 : gpus;
        replicas_.assign((size_t)n, nullptr);
        std::vector<std::string> errors((size_t)n);
        auto create = [&](int g) {
            const float origin[3] = {0.0f, -1.0f, 0.0f}, light[3] = {-1.0f, -3.0f, 2.0f}, eye[3] = {0.0f, 0.0f, -4.0f};
            if (n > 1 && set_device(g) != RT_OK) {
                errors[(size_t)g] = std::string("cudaSetDevice: ") + rt_last_error();
                return;
            }
            if (rt_scene_create(level, origin, 1.0f, light, eye, &replicas_[(size_t)g]) != RT_OK)
                errors[(size_t)g] = std::string("Scene::default: ") + rt_last_error();  // (the error text is thread-local)
        };
        if (n == 1) {
            create(0);
        } else {
            std::vector<std::thread> workers;
            for (int g = 0; g < n; g++) workers.emplace_back(create, g);
            for (std::thread &t : workers) t.join();
            set_device(0);
        }
        for (const std::string &e : errors)
            if (!e.empty()) {
                for (rt_scene *s : replicas_) rt_scene_destroy(s);
                replicas_.clear();
                throw Panic(e);
            }
    }
    ~Scene() {
        for (rt_scene *s : replicas_) rt_scene_destroy(s);
    }
    Scene(const Scene &) = delete;
    Scene &operator=(const Scene &) = delete;
    int gpus() const { return (int)replicas_.size(); }
    rt_scene *const *replicas() const { return replicas_.data(); }

  private:
    static int set_device(int g) { return rt_set_device(g); }
    std::vector<rt_scene *> replicas_;
};

struct Renderer {
    // render.rs:260-310.  `camera` (extension) may be NULL.  Sizes need not be
    // multiples of 64 (the reference asserts they are, render.rs:265-266).
    static void render(const RenderOptions &o, const Scene &scene, RGBABufferWriter &writer,
                       const rt_camera *camera = nullptr, rt_stats *stats = nullptr) {
        writer.begin(o.width, o.height);
        ImageRegion full;
        full.l = 0, full.r = o.width, full.b = 0, full.t = o.height;
        RGBABuffer frame(full);
        rt_check(rt_render_frame_multi(scene.replicas(), scene.gpus(), camera, o.width, o.height, o.samples_per_pixel,
                                       frame.data(), frame.len(), stats),
                 "Renderer::render");
        writer.write_rgba_buffer(frame);
    }

    // render.rs:218-255: the pixels of `buf.region()` (a bucket, or any window of the frame), row-major from
    // row b, on the scene's first GPU.  Same seam as the reference's, for callers that schedule regions
    // themselves (region-of-interest rendering, README "season 2").
    static void render_region(const RenderOptions &o, const Scene &scene, RGBABuffer &buf) {
        const ImageRegion &r = buf.region();
        rt_check(rt_render_region(scene.replicas()[0], o.width, o.height, o.samples_per_pixel, r.l, r.b, r.r, r.t,
                                  buf.data(), buf.len()),
                 "Renderer::render_region");
    }

    // Undersampled preview (README.md:42-48 "interactive rendering with undersampling"; extension): one traced
    // pixel per step x step block, handed to the writer as one full-size buffer.
    static void render_preview(const RenderOptions &o, const Scene &scene, RGBABufferWriter &writer, uint32_t step,
                               const rt_camera *camera = nullptr) {
        writer.begin(o.width, o.height);
        ImageRegion full;
        full.l = 0, full.r = o.width, full.b = 0, full.t = o.height;
        RGBABuffer frame(full);
        rt_check(rt_render_preview(scene.replicas()[0], camera, o.width, o.height, step, frame.data(), frame.len(), nullptr),
                 "Renderer::render_preview");
        writer.write_rgba_buffer(frame);
    }

    // The reference's own schedule (render.rs:265-309): the frame cut into 64x64 buckets, row-major y then x,
    // each rendered by render_region and handed to the writer as it completes.  Kept for conformance of the
    // writer seam (buckets "might be anywhere", render.rs:25-27) and selected by `rtrace --buckets`; render()
    // above is the fast path.  Like the reference it insists on multiples of 64.
    static void render_buckets(const RenderOptions &o, const Scene &scene, RGBABufferWriter &writer) {
        const uint16_t bucket = 64;
        if (o.width % bucket != 0) throw Panic("assertion failed: o.width % BUCKET_SIZE == 0");
        if (o.height % bucket != 0) throw Panic("assertion failed: o.height % BUCKET_SIZE == 0");
        writer.begin(o.width, o.height);
        for (uint32_t y = 0; y < o.height; y += bucket)
            for (uint32_t x = 0; x < o.width; x += bucket) {
                ImageRegion r;
                r.l = (uint16_t)x, r.r = (uint16_t)(x + bucket), r.b = (uint16_t)y, r.t = (uint16_t)(y + bucket);
                RGBABuffer buf(r);
                render_region(o, scene, buf);
                writer.write_rgba_buffer(buf);
            }
    }

    // A sweep of frames (extension; BASELINE configs[4]): the scene's GPUs draw frames from one queue, every GPU pipelines its
    // own frames (copy-out of one frame overlapping the render of the next two), and `sink(f, bytes, len)` is
    // called once per frame, in frame order, on the calling thread -- the role of the reference's main thread
    // draining the channel into the writer (render.rs:301-307).  With rgb = true the frames arrive as RGB8
    // (the body of the P6 file, alpha already dropped).  An exception thrown by the sink is rethrown here once the
    // sweep has returned (sweep_through).
    template <class Sink>
    static void render_sweep(const RenderOptions &o, const Scene &scene, const std::vector<rt_camera> &cameras,
                             Sink &&sink, rt_stats *stats = nullptr, bool rgb = false) {
        sweep_through(sink, "Renderer::render_sweep", [&](rt_frame_callback cb, void *user) {
            return rt_render_sweep_multi(scene.replicas(), scene.gpus(), cameras.data(), (uint32_t)cameras.size(), o.width,
                                         o.height, o.samples_per_pixel, rgb ? 1 : 0, cb, user, stats);
        });
    }

    // The same sweep delivering every frame as a PNG file encoded on its GPU (extension): `sink(f, file, len)`.
    template <class Sink>
    static void render_sweep_png(const RenderOptions &o, const Scene &scene, const std::vector<rt_camera> &cameras,
                                 Sink &&sink, rt_stats *stats = nullptr) {
        sweep_through(sink, "Renderer::render_sweep_png", [&](rt_frame_callback cb, void *user) {
            return rt_render_sweep_png(scene.replicas(), scene.gpus(), cameras.data(), (uint32_t)cameras.size(), o.width,
                                       o.height, o.samples_per_pixel, cb, user, stats);
        });
    }

    // The same sweep as one animated PNG whose frames each show for delay_num / delay_den seconds (extension):
    // `sink(f, payload, len)` in frame order, and the payloads written one after the other are the file.
    template <class Sink>
    static void render_sweep_apng(const RenderOptions &o, const Scene &scene, const std::vector<rt_camera> &cameras,
                                  uint16_t delay_num, uint16_t delay_den, Sink &&sink, rt_stats *stats = nullptr) {
        sweep_through(sink, "Renderer::render_sweep_apng", [&](rt_frame_callback cb, void *user) {
            return rt_render_sweep_apng(scene.replicas(), scene.gpus(), cameras.data(), (uint32_t)cameras.size(), o.width,
                                        o.height, o.samples_per_pixel, delay_num, delay_den, cb, user, stats);
        });
    }

    // Which frame of an animated PNG render_png writes, and the animation's frame count and frame delay.
    struct ApngFrame {
        uint32_t frame, n_frames;
        uint16_t delay_num, delay_den;
    };

    // One frame (or an undersampled preview when preview_step > 0) as a PNG file on `f` (extension): rendered into
    // device memory of the first GPU (with several GPUs their kernels store their rows there) and encoded there,
    // so only the file crosses the host link.  With `apng` the frame's payload of that animation is written instead.
    static void render_png(const RenderOptions &o, const Scene &scene, FILE *f, const rt_camera *camera = nullptr,
                           uint32_t preview_step = 0, rt_stats *stats = nullptr, const ApngFrame *apng = nullptr) {
        struct Buffers {
            void *frame = nullptr, *file = nullptr;
            ~Buffers() {
                rt_device_free(frame);
                rt_host_free(file);
            }
        } b;
        const size_t frame_bytes = (size_t)o.width * o.height * 4;
        size_t bound = 0, len = 0;
        rt_check(apng ? rt_apng_bound(o.width, o.height, apng->n_frames, &bound) : rt_png_bound(o.width, o.height, &bound),
                 "Renderer::render_png");
        rt_check(rt_device_alloc(frame_bytes, &b.frame), "Renderer::render_png");
        rt_check(rt_host_alloc(bound, &b.file), "Renderer::render_png");
        uint8_t *frame = static_cast<uint8_t *>(b.frame);
        if (preview_step)
            rt_check(rt_render_preview(scene.replicas()[0], camera, o.width, o.height, preview_step, frame, frame_bytes, nullptr),
                     "Renderer::render_preview");
        else
            rt_check(rt_render_frame_multi(scene.replicas(), scene.gpus(), camera, o.width, o.height, o.samples_per_pixel,
                                           frame, frame_bytes, stats),
                     "Renderer::render");
        uint8_t *file = static_cast<uint8_t *>(b.file);
        rt_check(apng ? rt_encode_apng_frame(frame, o.width, o.height, 0, apng->frame, apng->n_frames, apng->delay_num,
                                             apng->delay_den, file, bound, &len, nullptr)
                      : rt_encode_png(frame, o.width, o.height, 0, file, bound, &len, nullptr),
                 "Renderer::render_png");
        if (fwrite(b.file, 1, len, f) != len) throw Panic("write_all failed");
        fflush(f);
    }

    // One frame before quantisation as a colour PFM on `f` (extension): rendered on the scene's GPUs into pinned host
    // memory as float RGBA (rt_render_frame_multi_f32), then written by write_pfm.
    static void render_pfm(const RenderOptions &o, const Scene &scene, FILE *f, const rt_camera *camera = nullptr,
                           rt_stats *stats = nullptr) {
        struct Frame {
            void *p = nullptr;
            ~Frame() { rt_host_free(p); }
        } b;
        const size_t frame_bytes = (size_t)o.width * o.height * 16;
        rt_check(rt_host_alloc(frame_bytes, &b.p), "Renderer::render_pfm");
        float *frame = static_cast<float *>(b.p);
        rt_check(rt_render_frame_multi_f32(scene.replicas(), scene.gpus(), camera, o.width, o.height, o.samples_per_pixel,
                                           frame, frame_bytes, stats),
                 "Renderer::render_pfm");
        write_pfm(f, o.width, o.height, frame, (size_t)o.width * 4);
    }

  private:
    // `call(cb, user)` runs a sweep that hands each frame to `sink`.  An exception thrown by the sink does not cross
    // the C boundary: it is caught in the trampoline, the remaining frames are skipped, and it is rethrown here once
    // the sweep has returned (no render or copy is left in flight on the library's buffers).
    template <class Sink, class Call>
    static void sweep_through(Sink &sink, const char *what, Call &&call) {
        struct Ctx {
            Sink *sink;
            std::exception_ptr error;
        } ctx{&sink, nullptr};
        auto trampoline = [](void *user, uint32_t frame, const uint8_t *data, size_t len) {
            Ctx *c = static_cast<Ctx *>(user);
            if (c->error) return;  // a previous frame's sink failed: drain quietly
            try {
                (*c->sink)(frame, data, len);
            } catch (...) {
                c->error = std::current_exception();
            }
        };
        const int rc = call(trampoline, &ctx);
        if (ctx.error) std::rethrow_exception(ctx.error);
        rt_check(rc, what);
    }
};

}  // namespace sphere_tracer
