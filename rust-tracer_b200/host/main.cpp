// main.cpp -- the `rtrace` binary: same command line, environment, output format
// and exit behaviour as the reference (src/rust/main.rs), with the renderer
// running on B200 GPUs through librtrace_b200.so.
//
//   rtrace [--width=X] [--height=Y] [--samples-per-pixel=SAMPLES] [--num-cores N] <output>
//
// <output> is `-` (binary PPM on stdout) or a file that must be named *.tga and
// receives a binary PPM (main.rs:63-76, render.rs:373-383).  RTRACEMAXPROCS and
// --num-cores are still accepted (main.rs:24-29,56-61) so `RTRACEMAXPROCS=4 make
// image` keeps working; they size the reference's CPU thread pool, which no
// longer exists -- the GPU path ignores them.
// Additive flags: --level=L (scene depth, default 8 as at render.rs:147),
// --gpus=N / RTRACE_GPUS (default 1: one frame = interleaved row blocks over the GPUs; a sweep = the GPUs draw
// frames from one queue), --frames=K (orbit sweep; frame f goes to <stem>.f.tga, frame 0 is the reference camera), --stats (summary on stderr), --buckets (the reference's 64x64 bucket
// schedule through Renderer::render_region instead of one launch per frame), --format=tga|png|apng (a real TGA, a PNG
// encoded on the GPU: the output is then named *.png and sweep frames <stem>.f.png, or all frames in ONE animated PNG
// named *.png), --fps=F (frame rate of --format apng), --format=pfm (the pixels before quantisation as a colour PFM
// of 32-bit floats, named *.pfm; sweep frames <stem>.f.pfm).
#include <cerrno>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "render.hpp"

using namespace sphere_tracer;

namespace {

const char *USAGE =
    "rtrace 0.2.0\n"
    "Sebastian Thiel <byronimo@mail.com>\n"
    "A toy-raytracer for rendering a scene with spheres\n"
    "\n"
    "USAGE:\n"
    "    rtrace [OPTIONS] <output>\n"
    "\n"
    "FLAGS:\n"
    "    -h, --help       Prints help information\n"
    "    -V, --version    Prints version information\n"
    "\n"
    "OPTIONS:\n"
    "        --height <Y>                       The height of the output image [default: 1024]\n"
    "        --num-cores <numcores>             Amount of cores to do the rendering on [default: 1]\n"
    "                                           If this is not set, you may also use the RTRACEMAXPROCS\n"
    "                                           environment variable, e.g. RTRACEMAXPROCS=4.\n"
    "                                           The commandline always overrides environment variables.\n"
    "                                           (kept for compatibility: rendering runs on the GPU)\n"
    "        --samples-per-pixel <SAMPLES>      Amount of samples per pixel. 4 means 16 over-samples [default: 1]\n"
    "        --width <X>                        The width of the output image [default: 1024]\n"
    "        --level <L>                        Depth of the sphere pyramid [default: 8]\n"
    "        --gpus <N>                         GPUs to render on: a frame is split into interleaved row blocks,\n"
    "                                           a sweep (--frames) into whole frames [default: 1 or RTRACE_GPUS]\n"
    "        --frames <K>                       Render a K-frame orbit of the camera [default: 1]\n"
    "        --format <ppm|tga|png>             File contents: the reference's binary PPM, a real TGA, or a PNG encoded\n"
    "                                           on the GPU (the output is then named *.png) [default: ppm]\n"
    "        --format apng                      All frames in one animated PNG encoded on the GPU (named *.png)\n"
    "        --format pfm                       The unquantised pixels as a colour PFM of 32-bit floats (named *.pfm)\n"
    "        --fps <F>                          Frames per second of --format apng, 1..65535 [default: 24]\n"
    "        --preview <N>                      Undersampled preview: trace one pixel per NxN block (1 sample) [default: off]\n"
    "        --stats                            Print a timing summary to stderr\n"
    "        --buckets                          Render 64x64 buckets one by one in the reference's order (sizes must\n"
    "                                           be multiples of 64, as in the reference); default is whole frames\n"
    "\n"
    "ARGS:\n"
    "    <output>    Either a file with .tga extension (.png with --format png or apng, .pfm with --format pfm), or - to\n"
    "                write file to stdout\n";

[[noreturn]] void usage_error(const std::string &msg) {
    // clap 2: message + usage hint on stderr, exit status 1
    fprintf(stderr, "error: %s\n\nUSAGE:\n    rtrace [OPTIONS] <output>\n\nFor more information try --help\n", msg.c_str());
    exit(1);
}

// Rust's `str::parse::<uN>()`: optional leading '+', decimal digits only, range-checked.
bool parse_unsigned(const std::string &s, unsigned long long max, unsigned long long *out) {
    size_t i = 0;
    if (!s.empty() && s[0] == '+') i = 1;
    if (i >= s.size()) return false;
    unsigned long long v = 0;
    for (; i < s.size(); i++) {
        if (s[i] < '0' || s[i] > '9') return false;
        v = v * 10 + (unsigned)(s[i] - '0');
        if (v > max) return false;
    }
    *out = v;
    return true;
}

// `.parse().unwrap()` on a bad value panics (exit code 101), main.rs:56,79-81
unsigned long long parse_or_panic(const std::string &s, unsigned long long max, const char *what) {
    unsigned long long v = 0;
    if (!parse_unsigned(s, max, &v)) {
        fprintf(stderr, "thread 'main' panicked at 'called `Result::unwrap()` on an `Err` value: ParseIntError' (%s = '%s')\n", what, s.c_str());
        exit(101);
    }
    return v;
}

struct Args {
    std::string width, height, ssp, numcores, output, level, gpus, frames, format, preview, fps;
    bool has_output = false, stats = false, buckets = false;
};

Args parse_args(int argc, char **argv) {
    Args a;
    struct Opt {
        const char *name;
        std::string Args::*field;
    };
    const Opt opts[] = {{"--width", &Args::width},   {"--height", &Args::height}, {"--samples-per-pixel", &Args::ssp},
                        {"--num-cores", &Args::numcores}, {"--level", &Args::level},   {"--gpus", &Args::gpus},
                        {"--frames", &Args::frames}, {"--format", &Args::format},
                        {"--preview", &Args::preview}, {"--fps", &Args::fps}};
    bool only_positional = false;
    for (int i = 1; i < argc; i++) {
        std::string arg = argv[i];
        if (!only_positional && arg == "--") {
            only_positional = true;
            continue;
        }
        if (!only_positional && (arg == "-h" || arg == "--help")) {
            fputs(USAGE, stdout);
            exit(0);
        }
        if (!only_positional && (arg == "-V" || arg == "--version")) {
            puts("rtrace 0.2.0");
            exit(0);
        }
        if (!only_positional && arg == "--stats") {
            a.stats = true;
            continue;
        }
        if (!only_positional && arg == "--buckets") {
            a.buckets = true;
            continue;
        }
        if (!only_positional && arg.size() > 2 && arg[0] == '-' && arg[1] == '-') {
            bool matched = false;
            for (const Opt &o : opts) {
                size_t n = strlen(o.name);
                if (arg.compare(0, n, o.name) == 0 && (arg.size() == n || arg[n] == '=')) {
                    std::string value;
                    if (arg.size() == n) {  // `--flag value`
                        if (i + 1 >= argc) usage_error("The argument '" + std::string(o.name) + " <value>' requires a value but none was supplied");
                        value = argv[++i];
                    } else {
                        value = arg.substr(n + 1);
                    }
                    if (value.empty()) usage_error("The argument '" + std::string(o.name) + " <value>' requires a value but none was supplied");
                    a.*(o.field) = value;
                    matched = true;
                    break;
                }
            }
            if (!matched) usage_error("Found argument '" + arg + "' which wasn't expected, or isn't valid in this context");
            continue;
        }
        if (!only_positional && arg.size() > 1 && arg[0] == '-' && arg != "-")
            usage_error("Found argument '" + arg + "' which wasn't expected, or isn't valid in this context");
        if (a.has_output) usage_error("Found argument '" + arg + "' which wasn't expected, or isn't valid in this context");
        a.output = arg;
        a.has_output = true;
    }
    if (!a.has_output) usage_error("The following required arguments were not provided:\n    <output>");
    if (a.output.empty()) usage_error("The argument '<output>' requires a value but none was supplied");  // empty_values(false)
    return a;
}

// Path::extension(): the part after the last '.' of the file name, if the name does not start with it
std::string extension_of(const std::string &path) {
    size_t slash = path.find_last_of('/');
    std::string name = slash == std::string::npos ? path : path.substr(slash + 1);
    size_t dot = name.find_last_of('.');
    if (dot == std::string::npos || dot == 0) return ".UNSET";
    return name.substr(dot + 1);
}

std::string with_extension(const std::string &path, const std::string &ext) {
    size_t slash = path.find_last_of('/');
    size_t start = slash == std::string::npos ? 0 : slash + 1;
    size_t dot = path.find_last_of('.');
    std::string stem = (dot == std::string::npos || dot <= start) ? path : path.substr(0, dot);
    return stem + "." + ext;
}

rt_camera orbit_camera(unsigned frame, unsigned n_frames) {
    // Extension (SURVEY F6): rotate the reference camera about the flake's vertical axis.
    const double th = 2.0 * M_PI * (double)frame / (double)n_frames;
    double c = cos(th), s = sin(th);
    if (frame % n_frames == 0) c = 1.0, s = 0.0;
    auto rot = [&](double x, double y, double z, float out[3]) {
        out[0] = (float)(c * x + s * z);
        out[1] = (float)y;
        out[2] = (float)(-s * x + c * z);
    };
    rt_camera cam;
    rot(0.0, 0.0, -4.0, cam.eye);
    rot(1.0, 0.0, 0.0, cam.right);
    cam.up[0] = 0.0f, cam.up[1] = 1.0f, cam.up[2] = 0.0f;
    rot(0.0, 0.0, 1.0, cam.forward);
    return cam;
}

}  // namespace

int main(int argc, char **argv) {
    // main.rs:24-29: RTRACEMAXPROCS, default 1, unparsable -> 1 (accepted, unused by the GPU path)
    unsigned long long nc_from_env = 1;
    if (const char *e = getenv("RTRACEMAXPROCS")) {
        unsigned long long v;
        if (parse_unsigned(e, ~0ull >> 1, &v)) nc_from_env = v;
    }
    Args args = parse_args(argc, argv);
    unsigned long long num_cores = parse_or_panic(args.numcores.empty() ? "1" : args.numcores, ~0ull >> 1, "num-cores");
    unsigned long long pool_threads = num_cores > 1 ? num_cores : nc_from_env;  // main.rs:57-61 (quirk kept)
    if (pool_threads == 0) {  // ThreadPool::new(0) asserts
        fprintf(stderr, "thread 'main' panicked at 'assertion failed: num_threads >= 1'\n");
        return 101;
    }

    // main.rs:63-76
    const std::string &output_file = args.output;
    FileOrAnyWriter output;
    FILE *fp = nullptr;
    const bool png = args.format == "png", apng = args.format == "apng", pfm = args.format == "pfm";
    const std::string ext = png || apng ? "png" : pfm ? "pfm" : "tga";
    // before the output's name is checked: a misused --fps is a usage error whatever the name
    if (!args.fps.empty() && !apng) usage_error("The argument '--fps' can only be used with '--format apng'");
    unsigned long long fps = 24;
    if (!args.fps.empty() && (!parse_unsigned(args.fps, 65535, &fps) || fps == 0))
        usage_error("Invalid value for '--fps <F>': '" + args.fps + "' is not a whole number in 1..65535");
    if (output_file != "-") {
        if (extension_of(output_file) != ext) {
            printf("Output file '%s' must have the %s extension, e.g. %s\n", output_file.c_str(), ext.c_str(), with_extension(output_file, ext).c_str());
            return 0;
        }
    }

    // main.rs:78-82
    RenderOptions options;
    options.width = (uint16_t)parse_or_panic(args.width.empty() ? "1024" : args.width, 65535, "width");
    options.height = (uint16_t)parse_or_panic(args.height.empty() ? "1024" : args.height, 65535, "height");
    options.samples_per_pixel = (uint16_t)parse_or_panic(args.ssp.empty() ? "1" : args.ssp, 65535, "ssp");
    unsigned level = (unsigned)parse_or_panic(args.level.empty() ? "8" : args.level, 12, "level");
    const char *genv = getenv("RTRACE_GPUS");
    int gpus = (int)parse_or_panic(!args.gpus.empty() ? args.gpus : (genv && *genv ? genv : "1"), 64, "gpus");
    unsigned frames = (unsigned)parse_or_panic(args.frames.empty() ? "1" : args.frames, 100000, "frames");
    if (gpus < 1) gpus = 1;
    if (frames < 1) frames = 1;
    if (!args.format.empty() && args.format != "ppm" && args.format != "tga" && !png && !apng && !pfm)
        usage_error("'" + args.format + "' isn't a valid value for '--format <ppm|tga|png|apng|pfm>'");
    // the bucket schedule exists to drive the host writer seam; a PNG is encoded on the GPU from a whole frame,
    // and a PFM is the float frame of the whole-frame path
    if ((png || apng || pfm) && args.buckets) usage_error("The argument '--buckets' cannot be used with '--format " + args.format + "'");
    if (pfm && !args.preview.empty()) usage_error("The argument '--preview' cannot be used with '--format pfm'");
    const bool real_tga = args.format == "tga";
    const unsigned preview = args.preview.empty() ? 0u : (unsigned)parse_or_panic(args.preview, 1024, "preview");
    if (options.width == 0 || options.height == 0) {
        fprintf(stderr, "thread 'main' panicked at 'width and height must be at least 1'\n");
        return 101;
    }

    try {
        using clk = std::chrono::steady_clock;
        auto t0 = clk::now();
        Scene scene(level, gpus);  // Arc::new(Scene::default()), main.rs:23
        auto t1 = clk::now();
        double render_ms = 0.0, kernel_ms = 0.0;
        auto frame_path = [&](unsigned f) {
            if (frames == 1 || output_file == "-" || apng) return output_file;
            char suffix[32];
            snprintf(suffix, sizeof(suffix), "%04u.%s", f, ext.c_str());
            return with_extension(output_file, suffix);
        };
        auto open_output = [&](unsigned f) {
            if (output_file == "-") return FileOrAnyWriter::any_writer_stdout();
            fp = fopen(frame_path(f).c_str(), "wb");  // fs::File::create(&p).unwrap()
            if (!fp) throw Panic(std::string("called `Result::unwrap()` on an `Err` value: ") + strerror(errno));
            return FileOrAnyWriter::file_writer(fp);
        };
        if (frames > 1 && !preview && !args.buckets && !pfm) {
            // orbit sweep: the GPUs draw frames from one queue, copy-out of a frame overlapping the render of the next ones;
            // the frames come back in order (rt_render_sweep_multi)
            std::vector<rt_camera> cams;
            for (unsigned f = 0; f < frames; f++) cams.push_back(orbit_camera(f, frames));
            rt_stats st;
            auto r0 = clk::now();
            if (apng) {  // frames arrive as the animation's payloads, in order: one file
                output = open_output(0);
                Renderer::render_sweep_apng(options, scene, cams, 1, (uint16_t)fps, [&](uint32_t, const uint8_t *data, size_t len) {
                    if (fwrite(data, 1, len, output.f) != len) throw Panic("write_all failed");
                }, &st);
                fflush(output.f);
                if (fp) fclose(fp), fp = nullptr;
            } else if (png) {  // frames arrive as complete PNG files
                Renderer::render_sweep_png(options, scene, cams, [&](uint32_t f, const uint8_t *file, size_t len) {
                    output = open_output(f);
                    if (fwrite(file, 1, len, output.f) != len) throw Panic("write_all failed");
                    fflush(output.f);
                    if (fp) fclose(fp), fp = nullptr;
                }, &st);
            } else {
                // frames arrive as RGB8: exactly the body PPMStdoutRGBABufferWriter would write (render.rs:377-397)
                Renderer::render_sweep(options, scene, cams, [&](uint32_t f, const uint8_t *rgb, size_t len) {
                    output = open_output(f);
                    if (real_tga) {
                        write_tga(output.f, options.width, options.height, rgb, (size_t)options.width * 3, 3);
                    } else {
                        fprintf(output.f, "P6\n%u %u\n255\n", (unsigned)options.width, (unsigned)options.height);
                        if (fwrite(rgb, 1, len, output.f) != len) throw Panic("write_all failed");
                        fflush(output.f);
                    }
                    if (fp) fclose(fp), fp = nullptr;
                }, &st, true);
            }
            render_ms += std::chrono::duration<double, std::milli>(clk::now() - r0).count();
            kernel_ms = 0.0;
        } else {
            for (unsigned f = 0; f < frames; f++) {
                if (!apng || f == 0) output = open_output(f);  // an animation is one file
                rt_camera cam = orbit_camera(f, frames);
                rt_stats st;
                if (pfm) {  // <stem>.f.pfm per frame, or the frames back to back on stdout
                    auto r0 = clk::now();
                    Renderer::render_pfm(options, scene, output.f, frames > 1 ? &cam : nullptr, &st);
                    render_ms += std::chrono::duration<double, std::milli>(clk::now() - r0).count();
                    kernel_ms += st.kernel_ms;
                } else if (png || apng) {
                    const Renderer::ApngFrame af{f, frames, 1, (uint16_t)fps};
                    auto r0 = clk::now();
                    Renderer::render_png(options, scene, output.f, frames > 1 ? &cam : nullptr, preview, &st, apng ? &af : nullptr);
                    render_ms += std::chrono::duration<double, std::milli>(clk::now() - r0).count();
                    kernel_ms += preview ? 0.0 : st.kernel_ms;
                } else {
                    std::unique_ptr<RGBABufferWriter> sink;
                    if (real_tga) sink.reset(new TGARGBABufferWriter(&output));
                    else sink.reset(new PPMStdoutRGBABufferWriter(true, &output));
                    RGBABufferWriter &writer = *sink;
                    auto r0 = clk::now();
                    if (preview) Renderer::render_preview(options, scene, writer, preview, frames > 1 ? &cam : nullptr);
                    else if (args.buckets) Renderer::render_buckets(options, scene, writer);  // the reference's 64x64 schedule
                    else Renderer::render(options, scene, writer, frames > 1 ? &cam : nullptr, &st);
                    render_ms += std::chrono::duration<double, std::milli>(clk::now() - r0).count();
                    kernel_ms += st.kernel_ms;
                }  // final write on drop (render.rs:331-335)
                if (fp && (!apng || f + 1 == frames)) fclose(fp), fp = nullptr;
            }
        }
        if (args.stats) {
            double scene_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
            double total_ms = std::chrono::duration<double, std::milli>(clk::now() - t0).count();
            double mpx = (double)options.width * options.height * frames / 1e6;
            // kernel time is only separable for single frames; a sweep overlaps render, copy and file writes
            const double basis_ms = kernel_ms > 0.0 ? kernel_ms : render_ms;
            fprintf(stderr,
                    "rtrace-b200: %ux%u spp %u level %u, %u frame(s) on %d GPU(s): scene %.2f ms, kernel %.3f ms, "
                    "render+write %.2f ms, total %.2f ms, %.1f Mpixel/s, %.1f Msample/s (%s)\n",
                    (unsigned)options.width, (unsigned)options.height, (unsigned)options.samples_per_pixel, level, frames, gpus,
                    scene_ms, kernel_ms, render_ms, total_ms, mpx / (basis_ms * 1e-3),
                    mpx * options.samples_per_pixel * options.samples_per_pixel / (basis_ms * 1e-3),
                    kernel_ms > 0.0 ? "kernel only" : "render + copy + file write, overlapped");
        }
    } catch (const Panic &p) {
        fprintf(stderr, "thread 'main' panicked at '%s'\n", p.what());
        return 101;
    }
    return 0;  // process::exit(0), main.rs:89
}
