// selftest.cpp -- the reference's own host-side tests of the render module (src/rust/render.rs:437-499),
// transcribed for the C++ mirror in render.hpp, plus the sink's progressive-rewrite rule.
//
//   rtrace_selftest basic_rendering   render.rs:466-481: 64x128, 2x2 samples, DummyWriter -> begin() called,
//                                     exactly 2 bucket writes (through Renderer::render_buckets, the
//                                     reference's 64x64 schedule); also one write for Renderer::render
//   rtrace_selftest image_region      render.rs:483-499
//   rtrace_selftest progressive PATH  render.rs:426-432: a file sink rewrites the whole image when a buffer
//                                     arrives and no write happened yet or the last one is >= 1 s old;
//                                     final write on drop (render.rs:331-335)
//   rtrace_selftest sink_error        an exception thrown by a sweep sink is rethrown after the sweep returns
//
// Prints one "ok ..." line per check and exits 0; any failure prints "FAILED ..." and exits 1.
#include <sys/stat.h>
#include <thread>

#include "render.hpp"

using namespace sphere_tracer;

namespace {

int failures = 0;
#define CHECK(cond)                                                        \
    do {                                                                   \
        if (!(cond)) {                                                     \
            fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); \
            failures++;                                                    \
        }                                                                  \
    } while (0)

// render.rs:448-461
struct DummyWriter : RGBABufferWriter {
    bool begin_called = false;
    unsigned write_rgba_buffer_count = 0;
    uint16_t w = 0, h = 0;
    std::vector<ImageRegion> regions;
    void begin(uint16_t x, uint16_t y) override {
        begin_called = true;
        w = x, h = y;
    }
    void write_rgba_buffer(const RGBABuffer &b) override {
        write_rgba_buffer_count += 1;
        regions.push_back(b.region());
    }
};

void basic_rendering() {
    RenderOptions o;
    o.width = 64, o.height = 128, o.samples_per_pixel = 2;  // render.rs:469-473
    Scene scene;
    DummyWriter w;
    Renderer::render_buckets(o, scene, w);
    CHECK(w.begin_called);                     // render.rs:479
    CHECK(w.write_rgba_buffer_count == 2);     // render.rs:480
    CHECK(w.w == 64 && w.h == 128);
    CHECK(w.regions.size() == 2 && w.regions[0].b == 0 && w.regions[0].t == 64 && w.regions[1].b == 64 && w.regions[1].t == 128);
    DummyWriter whole;
    Renderer::render(o, scene, whole);         // the GPU schedule: the frame arrives as one buffer
    CHECK(whole.begin_called && whole.write_rgba_buffer_count == 1);
    // sizes that are not multiples of 64 panic in the bucket schedule, as in the reference (render.rs:265-266)
    o.height = 100;
    bool panicked = false;
    try {
        DummyWriter w2;
        Renderer::render_buckets(o, scene, w2);
    } catch (const Panic &) {
        panicked = true;
    }
    CHECK(panicked);
    printf("ok basic_rendering\n");
}

void image_region() {
    ImageRegion r;  // render.rs:485-498, value for value
    r.l = 2, r.t = 18, r.r = 34, r.b = 2;
    CHECK(r.width() == 32);
    CHECK(r.height() == 16);
    CHECK(r.area() == 16 * 32);
    CHECK(r.contains(r));
    ImageRegion l = r;
    l.l = 1;
    CHECK(l.contains(r));
    CHECK(!r.contains(l));
    CHECK(r.buffer_offset(4, 5) == 3 * 32 + 2);  // render.rs:66-71
    printf("ok image_region\n");
}

off_t file_size(const char *path) {
    struct stat st;
    return stat(path, &st) == 0 ? st.st_size : -1;
}

std::vector<uint8_t> slurp(const char *path) {
    std::vector<uint8_t> v;
    FILE *f = fopen(path, "rb");
    if (!f) return v;
    uint8_t buf[4096];
    size_t n;
    while ((n = fread(buf, 1, sizeof(buf), f)) > 0) v.insert(v.end(), buf, buf + n);
    fclose(f);
    return v;
}

void progressive(const char *path) {
    const uint16_t W = 8, H = 4;
    const size_t hdr = strlen("P6\n8 4\n255\n"), full = hdr + (size_t)W * H * 3;
    FILE *fp = fopen(path, "wb");
    CHECK(fp != nullptr);
    FileOrAnyWriter out = FileOrAnyWriter::file_writer(fp);
    auto band = [&](uint16_t row, uint8_t value) {
        ImageRegion r;
        r.l = 0, r.r = W, r.b = row, r.t = (uint16_t)(row + 1);
        std::unique_ptr<RGBABuffer> b(new RGBABuffer(r));
        memset(b->data(), value, b->len());
        return b;
    };
    auto pixel = [&](const std::vector<uint8_t> &file, unsigned row) { return file.size() >= full ? file[hdr + (size_t)row * W * 3] : 0xEE; };
    {
        PPMStdoutRGBABufferWriter sink(true, &out);
        sink.begin(W, H);
        CHECK(file_size(path) == 0);                      // begin() writes nothing
        sink.write_rgba_buffer(*band(0, 10));
        CHECK((size_t)file_size(path) == full);           // first buffer: flushed right away (render.rs:427-428)
        CHECK(pixel(slurp(path), 0) == 10);
        sink.write_rgba_buffer(*band(1, 20));             // < 1 s after the last write: kept in memory only
        CHECK(pixel(slurp(path), 1) != 20);
        std::this_thread::sleep_for(std::chrono::milliseconds(1100));
        sink.write_rgba_buffer(*band(2, 30));             // >= 1 s later: the whole image is rewritten
        std::vector<uint8_t> f = slurp(path);
        CHECK(f.size() == full && pixel(f, 1) == 20 && pixel(f, 2) == 30);
        sink.write_rgba_buffer(*band(3, 40));             // again within the second
        CHECK(pixel(slurp(path), 3) != 40);
    }  // drop: final write (render.rs:331-335)
    fclose(fp);
    std::vector<uint8_t> f = slurp(path);
    CHECK(f.size() == full && memcmp(f.data(), "P6\n8 4\n255\n", hdr) == 0);
    CHECK(pixel(f, 0) == 10 && pixel(f, 1) == 20 && pixel(f, 2) == 30 && pixel(f, 3) == 40);
    // stdout-style sink (not a file): nothing is written before the drop
    FILE *fp2 = fopen(path, "wb");
    FileOrAnyWriter any{fp2, false};
    {
        PPMStdoutRGBABufferWriter sink(true, &any);
        sink.begin(W, H);
        sink.write_rgba_buffer(*band(0, 7));
        fflush(fp2);
        CHECK(file_size(path) == 0);
    }
    fclose(fp2);
    CHECK((size_t)file_size(path) == full);
    printf("ok progressive\n");
}

void sink_error() {
    RenderOptions o;
    o.width = 64, o.height = 32, o.samples_per_pixel = 1;
    Scene scene;
    std::vector<rt_camera> cams(5);
    for (rt_camera &c : cams) {
        memset(&c, 0, sizeof(c));
        c.eye[2] = -4.0f, c.right[0] = 1.0f, c.up[1] = 1.0f, c.forward[2] = 1.0f;
    }
    unsigned calls = 0;
    bool caught = false;
    try {
        Renderer::render_sweep(o, scene, cams, [&](uint32_t f, const uint8_t *, size_t) {
            calls++;
            if (f == 1) throw Panic("sink failed");
        });
    } catch (const Panic &p) {
        caught = std::string(p.what()) == "sink failed";
    }
    CHECK(caught && calls == 2);  // frames after the failing one are not handed to the sink
    // the scene is usable afterwards (nothing was left in flight)
    unsigned again = 0;
    Renderer::render_sweep(o, scene, cams, [&](uint32_t, const uint8_t *, size_t) { again++; });
    CHECK(again == 5);
    printf("ok sink_error\n");
}

// write_pfm on a synthetic 3x2 frame, no GPU: pixel (x, y) component c = ((y * 3 + x) * 4 + c) / 7 in f32, with a
// pitch of 5 pixels so that the writer must follow the stride.  Writes the colour PFM to `path` and the greyscale one
// of component 3 (the Pf variant, as `rtrace --aov` writes coverage and distance) to `path`.grey.pfm.
// tests/test_f32.py and tests/test_aov.py check the files' bytes.
void pfm(const char *path) {
    const uint16_t w = 3, h = 2;
    const size_t stride = 5 * 4;
    std::vector<float> px(stride * h, -1.0f);
    for (uint32_t y = 0; y < h; y++)
        for (uint32_t x = 0; x < w; x++)
            for (uint32_t c = 0; c < 4; c++) px[y * stride + x * 4 + c] = (float)((y * w + x) * 4 + c) / 7.0f;
    FILE *f = fopen(path, "wb");
    if (!f) throw Panic(std::string("cannot create ") + path);
    write_pfm(f, w, h, px.data(), stride);
    fclose(f);
    const std::string grey = std::string(path) + ".grey.pfm";
    f = fopen(grey.c_str(), "wb");
    if (!f) throw Panic("cannot create " + grey);
    write_pfm(f, w, h, px.data() + 3, stride, 4, 1);
    fclose(f);
    printf("ok pfm\n");
}

}  // namespace

int main(int argc, char **argv) {
    const std::string what = argc > 1 ? argv[1] : "all";
    try {
        if (what == "image_region" || what == "all") image_region();
        if (what == "basic_rendering" || what == "all") basic_rendering();
        if (what == "sink_error" || what == "all") sink_error();
        if (what == "progressive" || what == "all") progressive(argc > 2 ? argv[2] : "/tmp/rtrace_selftest.tga");
        if (what == "pfm" || what == "all") pfm(argc > 2 ? argv[2] : "/tmp/rtrace_selftest.pfm");
    } catch (const Panic &p) {
        fprintf(stderr, "FAILED: panicked at '%s'\n", p.what());
        return 1;
    }
    return failures ? 1 : 0;
}
