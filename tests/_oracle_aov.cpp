// _oracle_aov.cpp -- the CPU oracle's AOV pixels (include/rtrace.h "geometry output").  TEST INFRASTRUCTURE ONLY.
//
// Built by tests/_oracle_aov.py into a library of its own, with oracle/Makefile's flags (FP contraction off, no
// fast-math).  The pinned oracle (oracle/oracle_rt.cpp) is included whole and unchanged, so the scene, the traversal
// (group_intersect from Hit::missed(), as Renderer::raytrace starts it) and the ray generation's arithmetic are its
// own code; what is added is render_pixel's sample loop keeping the geometry of each primary hit instead of the
// colour.  tests/_aov_ref.py ties it to the pinned library's orc_render_region kinds and orc_trace_rays hits
// (tests/test_aov.py).
#include "oracle_rt.cpp"

namespace {

// The AOV pixel (include/rtrace.h "geometry output"): render_pixel's rays, each traced from a miss as raytrace does
// (render.rs:188-189); no shadow ray.  v receives {nx, ny, nz, coverage, distance, px, py, pz}.
void aov_pixel(const orc_scene &s, const orc_camera *cam, uint32_t W, uint32_t H, uint32_t spp, uint32_t x, uint32_t y,
               float *v, Counters &k) {
    RFloat ssf = (RFloat)spp;
    RFloat total_recip = recip(ssf * ssf);
    RFloat width = (RFloat)W, height = (RFloat)H;
    Ray ray;
    ray.pos = cam ? Vector{cam->eye[0], cam->eye[1], cam->eye[2]} : s.eye;
    Vector n{0.0f, 0.0f, 0.0f}, pos{0.0f, 0.0f, 0.0f};
    RFloat cnt = 0.0f, dmin = INF;
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
            Hit h{INF, {0.0f, 0.0f, 0.0f}};
            group_intersect(*s.group, h, ray, k);
            if (h.has_missed()) continue;
            n = add(n, h.pos);  // h.pos is the unit normal (primitive.rs:83)
            cnt = cnt + 1.0f;
            if (h.distance < dmin) {
                dmin = h.distance;
                pos = add(ray.pos, mulfed(ray.dir, h.distance));  // render.rs:199, first term
            }
        }
    }
    n = mulfed(n, total_recip);
    const float out[8] = {n.x, n.y, n.z, cnt * total_recip, dmin, pos.x, pos.y, pos.z};
    memcpy(v, out, sizeof(out));
}

}  // namespace

extern "C" {

// The AOV frame: aov_out receives row_count * width * 8 floats {nx, ny, nz, coverage, distance, px, py, pz}, row j
// being image row row_start + j * row_stride; rows are shared out over nthreads threads.
void orc_render_rows_aov(const orc_scene *s, const orc_camera *cam, uint32_t width, uint32_t height, uint32_t spp,
                         uint32_t row_start, uint32_t row_stride, uint32_t row_count, uint32_t nthreads,
                         float *aov_out) {
    if (nthreads < 1) nthreads = 1;
    std::atomic<uint32_t> next(0);
    auto worker = [&]() {
        Counters k;
        for (uint32_t j; (j = next.fetch_add(1)) < row_count;) {
            const uint32_t y = row_start + j * row_stride;
            for (uint32_t x = 0; x < width; x++)
                aov_pixel(*s, cam, width, height, spp, x, y, aov_out + ((size_t)j * width + x) * 8, k);
        }
    };
    std::vector<std::thread> th;
    for (uint32_t i = 1; i < nthreads; i++) th.emplace_back(worker);
    worker();
    for (auto &t : th) t.join();
}

}  // extern "C"
