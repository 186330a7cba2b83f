// _oracle_f32.cpp -- the CPU oracle's pixel values before quantisation.  TEST INFRASTRUCTURE ONLY.
//
// Built by tests/_oracle_f32.py into a library of its own, with oracle/Makefile's flags (FP contraction off, no
// fast-math).  The pinned oracle (oracle/oracle_rt.cpp) is included whole and unchanged, so the scene, the
// traversal and Renderer::raytrace are its own code; what is added is render_pixel (oracle_rt.cpp) stopped
// before the quantisation.  The tests check that quantising these values gives orc_render_rows' bytes and the
// reference's shipped image (tests/test_f32.py), which ties this loop to the pinned one.
#include "oracle_rt.cpp"

namespace {

// render.rs:231-250: render_pixel's sample loop up to, and without, the quantisation (render.rs:92-109).
void accumulate_pixel(const orc_scene &s, const orc_camera *cam, uint32_t W, uint32_t H, uint32_t spp, uint32_t x,
                      uint32_t y, float *v, Counters &k, TraceStats &ts) {
    RFloat ssf = (RFloat)spp;
    RFloat total_recip = recip(ssf * ssf);
    RFloat width = (RFloat)W, height = (RFloat)H;
    Ray ray;
    ray.pos = cam ? Vector{cam->eye[0], cam->eye[1], cam->eye[2]} : s.eye;
    Vector g{0.0f, 0.0f, 0.0f};
    RFloat alpha = 0.0f;
    for (uint32_t ssx = 0; ssx < spp; ssx++) {
        for (uint32_t ssy = 0; ssy < spp; ssy++) {
            RFloat xres = (RFloat)x + (RFloat)ssx / ssf;
            RFloat yres = (RFloat)y + (RFloat)ssy / ssf;
            Vector d;
            d.x = xres - width / 2.0f;
            d.y = (height - yres) - height / 2.0f;
            d.z = width;
            if (cam) {  // camera extension, as in render_pixel
                Vector w;
                w.x = cam->right[0] * d.x + cam->up[0] * d.y + cam->forward[0] * d.z;
                w.y = cam->right[1] * d.x + cam->up[1] * d.y + cam->forward[1] * d.z;
                w.z = cam->right[2] * d.x + cam->up[2] * d.y + cam->forward[2] * d.z;
                d = w;
            }
            ray.dir = normalized(d);
            alpha += raytrace(s, ray, g, k, ts, nullptr);
        }
    }
    g = mulfed(g, total_recip);
    alpha *= total_recip;
    v[0] = g.x;
    v[1] = g.y;
    v[2] = g.z;
    v[3] = alpha;
}

}  // namespace

extern "C" {

// orc_render_rows without the quantisation: rgba_out receives row_count * width * 4 floats {r, g, b, alpha}, row j
// being image row row_start + j * row_stride; rows are shared out over nthreads threads.
void orc_render_rows_f32(const orc_scene *s, const orc_camera *cam, uint32_t width, uint32_t height, uint32_t spp,
                         uint32_t row_start, uint32_t row_stride, uint32_t row_count, uint32_t nthreads,
                         float *rgba_out, orc_counters *ctr) {
    if (nthreads < 1) nthreads = 1;
    std::atomic<uint32_t> next(0);
    std::vector<Counters> ks(nthreads);
    std::vector<TraceStats> tss(nthreads);
    auto worker = [&](uint32_t tid) {
        for (uint32_t j; (j = next.fetch_add(1)) < row_count;) {
            const uint32_t y = row_start + j * row_stride;
            for (uint32_t x = 0; x < width; x++)
                accumulate_pixel(*s, cam, width, height, spp, x, y, rgba_out + ((size_t)j * width + x) * 4, ks[tid],
                                 tss[tid]);
        }
    };
    std::vector<std::thread> th;
    for (uint32_t i = 1; i < nthreads; i++) th.emplace_back(worker, i);
    worker(0);
    for (auto &t : th) t.join();
    for (uint32_t i = 0; i < nthreads; i++) accumulate(ctr, ks[i], tss[i], 0);
    if (ctr) ctr->primary_rays += (uint64_t)width * row_count * spp * spp;
}

}  // extern "C"
