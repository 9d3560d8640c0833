// cli_main.cpp — `nr-ray-tracer render <scene> ...` on the B200 path: the call site of the boundary.
//
// Mirrors the reference CLI's render command (ray-tracer/src/commands/render.rs:104-115):
//   open output (create_new unless -f)  ->  load scene  ->  merge CLI/env camera over the file's camera
//   ->  build  ->  scene.render()  ->  gamma_correction(gamma)  ->  to_rgb8  ->  encode by extension
// Flags and NR_RT_CAMERA_* environment fallbacks follow ray-tracer/src/cli.rs:113-270 (field of view and defocus
// angle in degrees; image size needs exactly two of width / height / aspect ratio; default output out.png,
// default gamma 0.5).  Additions: --seed, --mode auto|pool|fused|wavefront|megakernel, --device N, --gpus N,
// --preview-every N, --adaptive-error REL [--adaptive-abs-error ABS] [--adaptive-min-samples N].
// Encoders available without external libraries: .png (stored/uncompressed deflate) and .ppm.
#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <unistd.h>

#include "../../include/nrrt.h"

[[noreturn]] static void die(const std::string& m) {
    std::fprintf(stderr, "Error: %s\n", m.c_str());
    std::exit(1);
}

// ---- argument parsers (cli.rs:71-110)
static bool parse_vector(const char* s, double out[3]) {
    // "x,y,z" with optional brackets / spaces
    std::string t;
    for (const char* p = s; *p; ++p)
        if (*p != '[' && *p != ']' && *p != '(' && *p != ')' && *p != ' ') t += *p;
    return std::sscanf(t.c_str(), "%lf,%lf,%lf", &out[0], &out[1], &out[2]) == 3;
}
static bool parse_aspect_ratio(const char* s, double* out) {
    double a, b;
    if (std::sscanf(s, "%lf:%lf", &a, &b) == 2 || std::sscanf(s, "%lf/%lf", &a, &b) == 2) {
        if (b == 0) return false;
        *out = a / b;
        return true;
    }
    char* e = nullptr;
    *out = std::strtod(s, &e);
    return e && *e == 0;
}

// ---- PNG (stored deflate) / PPM writers
static uint32_t crc_table[256];
static void crc_init() {
    for (uint32_t n = 0; n < 256; ++n) {
        uint32_t c = n;
        for (int k = 0; k < 8; ++k) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
        crc_table[n] = c;
    }
}
static uint32_t crc32(const uint8_t* p, size_t n, uint32_t c = 0xFFFFFFFFu) {
    for (size_t i = 0; i < n; ++i) c = crc_table[(c ^ p[i]) & 0xFF] ^ (c >> 8);
    return c;
}
static void put32(std::vector<uint8_t>& v, uint32_t x) {
    v.push_back(x >> 24), v.push_back(x >> 16), v.push_back(x >> 8), v.push_back(x);
}
static void chunk(FILE* f, const char* type, const std::vector<uint8_t>& data) {
    std::vector<uint8_t> hdr;
    put32(hdr, (uint32_t)data.size());
    std::fwrite(hdr.data(), 1, 4, f);
    std::vector<uint8_t> body(type, type + 4);
    body.insert(body.end(), data.begin(), data.end());
    std::fwrite(body.data(), 1, body.size(), f);
    std::vector<uint8_t> c;
    put32(c, crc32(body.data(), body.size()) ^ 0xFFFFFFFFu);
    std::fwrite(c.data(), 1, 4, f);
}
static void write_png(FILE* f, const uint8_t* rgb, uint32_t w, uint32_t h) {
    crc_init();
    const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    std::fwrite(sig, 1, 8, f);
    std::vector<uint8_t> ihdr;
    put32(ihdr, w), put32(ihdr, h);
    ihdr.push_back(8), ihdr.push_back(2), ihdr.push_back(0), ihdr.push_back(0), ihdr.push_back(0);
    chunk(f, "IHDR", ihdr);
    std::vector<uint8_t> raw;
    raw.reserve((size_t)h * (w * 3 + 1));
    for (uint32_t y = 0; y < h; ++y) {
        raw.push_back(0);  // filter: none
        raw.insert(raw.end(), rgb + (size_t)y * w * 3, rgb + (size_t)(y + 1) * w * 3);
    }
    std::vector<uint8_t> z;
    z.push_back(0x78), z.push_back(0x01);
    uint32_t a = 1, b = 0;
    for (size_t off = 0; off < raw.size() || off == 0;) {
        size_t n = raw.size() - off < 65535 ? raw.size() - off : 65535;
        bool last = off + n >= raw.size();
        z.push_back(last ? 1 : 0);
        z.push_back(n & 0xFF), z.push_back(n >> 8), z.push_back(~n & 0xFF), z.push_back((~n >> 8) & 0xFF);
        z.insert(z.end(), raw.begin() + off, raw.begin() + off + n);
        for (size_t i = 0; i < n; ++i) {
            a = (a + raw[off + i]) % 65521u;
            b = (b + a) % 65521u;
        }
        off += n;
        if (last) break;
    }
    put32(z, (b << 16) | a);
    chunk(f, "IDAT", z);
    chunk(f, "IEND", {});
}
static void write_ppm(FILE* f, const uint8_t* rgb, uint32_t w, uint32_t h) {
    std::fprintf(f, "P6\n%u %u\n255\n", w, h);
    std::fwrite(rgb, 1, (size_t)w * h * 3, f);
}
static void write_image(FILE* f, bool png, const uint8_t* rgb, uint32_t w, uint32_t h) {
    if (png) write_png(f, rgb, w, h);
    else write_ppm(f, rgb, w, h);
}
// Replaces `path` by a complete image: written to a temporary file next to it, then renamed over it, so that a viewer
// watching a progressive render never reads a half-written file.
static void replace_image(const std::string& path, bool png, const uint8_t* rgb, uint32_t w, uint32_t h) {
    const std::string tmp = path + ".tmp" + std::to_string((long)getpid());
    FILE* f = std::fopen(tmp.c_str(), "wb");
    if (!f) die("cannot open " + tmp + ": " + std::strerror(errno));
    write_image(f, png, rgb, w, h);
    const bool ok = std::fflush(f) == 0 && !std::ferror(f);
    if (std::fclose(f) != 0 || !ok || std::rename(tmp.c_str(), path.c_str()) != 0) {
        const std::string why = std::strerror(errno);
        std::remove(tmp.c_str());
        die("cannot write " + path + ": " + why);
    }
}

// A tolerance: a decimal number, whole string, finite and >= 0.
static bool parse_tolerance(const char* s, double* out) {
    char* e = nullptr;
    errno = 0;
    const double x = std::strtod(s, &e);
    if (!*s || !e || *e || errno || !std::isfinite(x) || !(x >= 0.0)) return false;
    *out = x;
    return true;
}

// Unsigned decimal integer, whole string, no sign, <= max (clap rejects "-1", "1e3", "" and overflow alike).
static bool parse_u64(const char* s, uint64_t max, uint64_t* out) {
    if (!s || !*s) return false;
    uint64_t x = 0;
    for (const char* p = s; *p; ++p) {
        if (*p < '0' || *p > '9') return false;
        const uint64_t dgt = (uint64_t)(*p - '0');
        if (x > (max - dgt) / 10) return false;
        x = x * 10 + dgt;
    }
    *out = x;
    return true;
}

static void usage() {
    std::puts(
        "Usage: nr-ray-tracer render [OPTIONS] <SCENE>\n"
        "       nr-ray-tracer create <cornell-box|cube|earth|noise|quads|triangles|spheres|simple-lights|convert-stl> [-o FILE] ...\n"
        "  -o, --output <FILE>            output file (.png or .ppm) [default: out.png]\n"
        "  -f, --force-overwrite          overwrite the output file\n"
        "      --gamma-value <G>          gamma [default: 0.5]\n"
        "  -W, --width <W>  -H, --height <H>  --aspect-ratio <R|W:H>      (exactly two, or none)\n"
        "      --background-color x,y,z  --look-at x,y,z  --look-from x,y,z  --view-up x,y,z\n"
        "      --field-of-view <DEG>  --defocus-angle <DEG>  --focus-distance <D>\n"
        "      --samples-per-pixel <N>  --ray-max-bounces <N>\n"
        "      --seed <N>  --mode auto|pool|fused|wavefront|megakernel  --device <N>\n"
        "      --gpus <N>                 render on GPUs device .. device+N-1 of this box (rows interleaved across them,\n"
        "                                 same image bit for bit; env NR_RT_GPUS)\n"
        "      --bvh reference|sah   reference = the reference's BVH (default), sah = surface-area-heuristic inner nodes\n"
        "      --preview-every <N>        render in passes and rewrite the output file whenever another N samples per\n"
        "                                 pixel are done (passes end on whole work chunks; the final image is the same;\n"
        "                                 one GPU only)\n"
        "      --adaptive-error <REL>     adaptive sampling: stop sampling a pixel once the estimated standard error of\n"
        "                                 its mean is at most ABS + REL x |mean| in every channel (0: every pixel takes\n"
        "                                 every sample; the image is then the same as without the flag; one GPU only)\n"
        "      --adaptive-abs-error <ABS> the absolute part of that tolerance (default 0)\n"
        "      --adaptive-min-samples <N> test a pixel only from N samples on (default: the first work-chunk boundary at\n"
        "                                 or above 1/8 of the samples per pixel).  Passes end at doubling chunk counts\n"
        "                                 from there, or as --preview-every sets them\n"
        "  -v, --verbose                  print timing\n"
        "Every camera option falls back to NR_RT_CAMERA_<NAME> (e.g. NR_RT_CAMERA_SAMPLES_PER_PIXEL).");
}

// `nr-ray-tracer create <kind> ...` (commands/create/*.rs): the scene generators are host-side authoring tools and
// live in the Python package (nr_ray_tracer_b200/create.py); this command hands its arguments over to them so the
// binary keeps the reference's two subcommands.  The package is found relative to the binary (bin/ -> package -> repo).
static int run_create(int argc, char** argv) {
    char self[4096];
    ssize_t n = readlink("/proc/self/exe", self, sizeof self - 1);
    if (n <= 0) die("cannot locate the executable");
    self[n] = 0;
    std::string root = self;
    for (int up = 0; up < 3; ++up) {
        size_t k = root.find_last_of('/');
        if (k == std::string::npos) die("cannot locate the Python package next to the executable");
        root.resize(k);
    }
    const char* old = std::getenv("PYTHONPATH");
    std::string pp = root + (old && *old ? std::string(":") + old : std::string());
    setenv("PYTHONPATH", pp.c_str(), 1);
    std::vector<char*> args;
    const char* py = std::getenv("NRRT_PYTHON");
    std::string python = py && *py ? py : "python3";
    args.push_back(const_cast<char*>(python.c_str()));
    args.push_back(const_cast<char*>("-m"));
    args.push_back(const_cast<char*>("nr_ray_tracer_b200.create"));
    for (int i = 2; i < argc; ++i) args.push_back(argv[i]);
    args.push_back(nullptr);
    execvp(args[0], args.data());
    die(std::string("cannot run ") + python + ": " + std::strerror(errno));
}

int main(int argc, char** argv) {
    if (argc < 2 || std::strcmp(argv[1], "--help") == 0 || std::strcmp(argv[1], "-h") == 0) {
        usage();
        return argc < 2 ? 2 : 0;
    }
    if (std::strcmp(argv[1], "create") == 0) return run_create(argc, argv);
    if (std::strcmp(argv[1], "render") != 0) die(std::string("unknown command '") + argv[1] + "' (commands: render, create)");
    std::string scene_path, output = "out.png", mode = "auto", bvh = "reference";
    bool force = false, verbose = false;
    float gamma = 0.5f;  // constants.rs:1
    uint64_t seed = 0, preview_every = 0, adaptive_min = 0;
    bool adaptive = false, adaptive_min_set = false, adaptive_abs_set = false;
    nrrt_adaptive_opts ad;
    std::memset(&ad, 0, sizeof ad);
    int device = 0, gpus = 1;
    if (const char* e = std::getenv("NR_RT_GPUS")) {
        uint64_t x = 0;
        if (!parse_u64(e, 64, &x) || x == 0) die("invalid value '" + std::string(e) + "' in NR_RT_GPUS");
        gpus = (int)x;
    }
    nrrt_camera_file cli;
    std::memset(&cli, 0, sizeof cli);

    auto set_camera = [&](const std::string& name, const char* val) -> bool {
        char* e = nullptr;
        auto u = [&](uint32_t& dst, uint32_t bit) {  // clap's u32 parser: digits only, no sign, must fit
            uint64_t x = 0;
            if (!parse_u64(val, 0xFFFFFFFFull, &x)) return false;
            dst = (uint32_t)x;
            cli.present |= bit;
            return true;
        };
        auto d = [&](double& dst, uint32_t bit) {
            if (!*val) return false;
            dst = std::strtod(val, &e);
            if (!e || *e) return false;
            cli.present |= bit;
            return true;
        };
        auto v = [&](double* dst, uint32_t bit) {
            if (!parse_vector(val, dst)) return false;
            cli.present |= bit;
            return true;
        };
        if (name == "width") return u(cli.width, NRRT_CAM_WIDTH);
        if (name == "height") return u(cli.height, NRRT_CAM_HEIGHT);
        if (name == "aspect-ratio") {
            if (!parse_aspect_ratio(val, &cli.aspect_ratio)) return false;
            cli.present |= NRRT_CAM_ASPECT_RATIO;
            return true;
        }
        if (name == "background-color") return v(cli.background, NRRT_CAM_BACKGROUND);
        if (name == "look-at") return v(cli.look_at, NRRT_CAM_LOOK_AT);
        if (name == "look-from") return v(cli.look_from, NRRT_CAM_LOOK_FROM);
        if (name == "view-up") return v(cli.view_up, NRRT_CAM_VIEW_UP);
        if (name == "field-of-view") return d(cli.field_of_view_deg, NRRT_CAM_FOV);
        if (name == "defocus-angle") return d(cli.defocus_angle_deg, NRRT_CAM_DEFOCUS);
        if (name == "focus-distance") return d(cli.focus_distance, NRRT_CAM_FOCUS);
        if (name == "samples-per-pixel") return u(cli.samples_per_pixel, NRRT_CAM_SPP);
        if (name == "ray-max-bounces") return u(cli.ray_max_bounces, NRRT_CAM_BOUNCES);
        if (name == "focal-length") return true;  // parsed, never used (cli.rs:229)
        return false;
    };
    const char* cam_names[] = {"width", "height", "aspect-ratio", "background-color", "look-at", "look-from", "view-up",
                               "focal-length", "field-of-view", "defocus-angle", "focus-distance", "samples-per-pixel",
                               "ray-max-bounces"};
    // environment first (clap: env is the fallback, flags win)
    for (const char* n : cam_names) {
        std::string env = "NR_RT_CAMERA_";
        for (const char* p = n; *p; ++p) env += (*p == '-') ? '_' : (char)toupper((unsigned char)*p);
        if (const char* v = std::getenv(env.c_str()))
            if (!set_camera(n, v)) die("invalid value '" + std::string(v) + "' in " + env);
    }
    for (int i = 2; i < argc; ++i) {
        std::string a = argv[i];
        auto need = [&]() -> const char* {
            if (i + 1 >= argc) die("missing value for " + a);
            return argv[++i];
        };
        if (a == "-h" || a == "--help") {
            usage();
            return 0;
        }
        if (a == "-f" || a == "--force-overwrite") force = true;
        else if (a == "-v" || a == "--verbose") verbose = true;
        else if (a == "-o" || a == "--output") output = need();
        else if (a == "--gamma-value") {
            const char* v = need();
            char* e = nullptr;
            gamma = std::strtof(v, &e);
            if (!*v || !e || *e) die("invalid value '" + std::string(v) + "' for --gamma-value");
        } else if (a == "--seed") {
            const char* v = need();
            if (!parse_u64(v, ~0ull, &seed)) die("invalid value '" + std::string(v) + "' for --seed");
        } else if (a == "--mode") mode = need();
        else if (a == "--bvh") bvh = need();
        else if (a == "--device") {
            const char* v = need();
            uint64_t x = 0;
            if (!parse_u64(v, 1023, &x)) die("invalid value '" + std::string(v) + "' for --device");
            device = (int)x;
        } else if (a == "--gpus") {
            const char* v = need();
            uint64_t x = 0;
            if (!parse_u64(v, 64, &x) || x == 0) die("invalid value '" + std::string(v) + "' for --gpus");
            gpus = (int)x;
        } else if (a == "--preview-every") {
            const char* v = need();
            if (!parse_u64(v, 0xFFFFFFFFull, &preview_every) || preview_every == 0)
                die("invalid value '" + std::string(v) + "' for --preview-every");
        } else if (a == "--adaptive-error") {
            const char* v = need();
            if (!parse_tolerance(v, &ad.rel_error)) die("invalid value '" + std::string(v) + "' for --adaptive-error");
            adaptive = true;
        } else if (a == "--adaptive-abs-error") {
            const char* v = need();
            if (!parse_tolerance(v, &ad.abs_error)) die("invalid value '" + std::string(v) + "' for --adaptive-abs-error");
            adaptive_abs_set = true;
        } else if (a == "--adaptive-min-samples") {
            const char* v = need();
            if (!parse_u64(v, 0xFFFFFFFFull, &adaptive_min))
                die("invalid value '" + std::string(v) + "' for --adaptive-min-samples");
            adaptive_min_set = true;
        }
        else if (a == "-W") { if (!set_camera("width", need())) die("invalid width"); }
        else if (a == "-H") { if (!set_camera("height", need())) die("invalid height"); }
        else if (a.rfind("--", 0) == 0) {
            std::string name = a.substr(2);
            bool known = false;
            for (const char* n : cam_names) known = known || name == n;
            if (!known) die("unknown option '" + a + "'");  // (without consuming the next argument)
            const char* v = need();
            if (!set_camera(name, v)) die("invalid value '" + std::string(v) + "' for " + a);
        } else if (a.size() > 1 && a[0] == '-') die("unknown option '" + a + "'"); else if (scene_path.empty()) scene_path = a;
        else die("unexpected argument '" + a + "'");
    }
    if (scene_path.empty()) die("missing <SCENE>");
    if (preview_every && gpus > 1)
        die("--preview-every renders on one GPU: it cannot be combined with --gpus " + std::to_string(gpus));
    if ((adaptive_abs_set || adaptive_min_set) && !adaptive)
        die(std::string(adaptive_abs_set ? "--adaptive-abs-error" : "--adaptive-min-samples") + " needs --adaptive-error");
    if (adaptive && gpus > 1)
        die("--adaptive-error renders on one GPU: it cannot be combined with --gpus " + std::to_string(gpus));
    auto ends = [&](const char* suf) {
        size_t n = std::strlen(suf);
        return output.size() >= n && output.compare(output.size() - n, n, suf) == 0;
    };
    const bool png = ends(".png"), ppm = ends(".ppm");
    if (!png && !ppm) die("unsupported output format (use .png or .ppm)");
    // ImageConfig::get_file (cli.rs:140-154): create_new unless -f
    FILE* out = std::fopen(output.c_str(), force ? "wb" : "wbx");
    if (!out) die("cannot open " + output + ": " + std::strerror(errno) + (force ? "" : " (use -f to overwrite)"));

    nrrt_loaded_scene* ls = nrrt_load_scene(scene_path.c_str(), nullptr);
    if (!ls) die(nrrt_load_last_error());
    nrrt_camera_file camf;
    nrrt_loaded_camera(ls, &camf);
    nrrt_camera_file_merge(&camf, &cli);  // render.rs:109
    nrrt_camera_config cfg;
    if (nrrt_camera_file_to_config(&camf, &cfg) != NRRT_OK) die("image size needs exactly two of --width / --height / --aspect-ratio");
    nrrt_camera cam;
    if (nrrt_host_camera_build(&cfg, &cam) != NRRT_OK) die("bad camera configuration");
    if (bvh != "reference" && bvh != "sah") die("--bvh must be reference or sah");
    nrrt_host_scene* hs = nrrt_host_build_ex(nrrt_loaded_graph(ls), bvh == "sah" ? NRRT_BUILD_SAH : NRRT_BUILD_REFERENCE);
    if (!hs) die(nrrt_host_last_error());
    nrrt_ctx* ctx = nullptr;  // device `device`: single-GPU render, and the output stage in every case
    if (nrrt_create(device, &ctx) != NRRT_OK) die(nrrt_last_error(nullptr));
    if (gpus == 1 && nrrt_scene_upload(ctx, nrrt_host_scene_desc(hs)) != NRRT_OK) die(nrrt_last_error(ctx));

    std::vector<float> image((size_t)cam.width * cam.height * 3);
    nrrt_render_opts opts;
    std::memset(&opts, 0, sizeof opts);
    opts.seed = seed;
    opts.world = 1;
    if (mode == "megakernel") opts.mode = NRRT_MODE_MEGAKERNEL;
    else if (mode == "wavefront") opts.mode = NRRT_MODE_WAVEFRONT;
    else if (mode == "fused") opts.mode = NRRT_MODE_FUSED;
    else if (mode == "pool") opts.mode = NRRT_MODE_POOL;
    else if (mode == "auto") opts.mode = NRRT_MODE_AUTO;
    else {
        std::fprintf(stderr, "error: unknown --mode '%s'\n", mode.c_str());
        return 2;
    }
    nrrt_render_stats st;
    auto t0 = std::chrono::steady_clock::now();
    // the reference draws a per-pixel progress bar (render.rs:48-59); with -v a percentage goes to stderr
    nrrt_progress_fn on_progress = [](uint64_t done, uint64_t total, void*) {
        std::fprintf(stderr, "\rrendering: %3u%%", total ? (unsigned)(done * 100 / total) : 100u);
        if (done >= total) std::fputc('\n', stderr);
    };
    if (gpus > 1) {  // one host thread + context per device inside the library, rows land in `image` directly
        std::vector<int> devs;
        for (int k = 0; k < gpus; ++k) devs.push_back(device + k);
        char msg[512] = "";
        if (nrrt_render_multi(devs.data(), gpus, nrrt_host_scene_desc(hs), &cam, &opts, image.data(),
                              verbose ? on_progress : nullptr, nullptr, &st, msg, sizeof msg) != NRRT_OK)
            die(msg);
    } else if (preview_every || adaptive) {
        // progressive: each pass renders up to the next multiple of N samples (rounded up to a chunk boundary), then the
        // image so far replaces the output file; the last pass completes the frame, which is nrrt_render's bit for bit.
        // Adaptive: the passes render the pixels still active only, and end at doubling chunk counts unless
        // --preview-every sets them; the frame is finished when no pixel is active.
        std::fclose(out);  // (opened above only for the create-new check: every image goes through replace_image)
        out = nullptr;
        nrrt_accum* acc = nullptr;
        const uint32_t spp = cam.samples_per_pixel ? cam.samples_per_pixel : 1;
        std::vector<uint32_t> starts(65);
        const uint32_t n_chunks = nrrt_chunk_starts(spp, (uint64_t)cam.width * cam.height, starts.data(), 65);
        uint32_t k = 1;  // chunk count the next adaptive pass ends on (without --preview-every)
        if (adaptive) {
            while (k < n_chunks && 8ull * starts[k] < spp) ++k;  // default: the first boundary at or above spp / 8
            ad.min_samples = adaptive_min_set ? (uint32_t)adaptive_min : starts[k];
            k = 1;
            while (k < n_chunks && starts[k] < ad.min_samples) ++k;
            if (nrrt_accum_create_adaptive(ctx, &cam, &opts, &ad, &acc) != NRRT_OK) die(nrrt_last_error(ctx));
        } else if (nrrt_accum_create(ctx, &cam, &opts, &acc) != NRRT_OK) {
            die(nrrt_last_error(ctx));
        }
        auto more = [&] { return adaptive ? nrrt_accum_active(acc) > 0 : nrrt_accum_samples(acc) < spp; };
        std::vector<uint8_t> preview(image.size());
        std::memset(&st, 0, sizeof st);
        while (more()) {
            uint64_t target;
            if (preview_every) {
                target = (nrrt_accum_samples(acc) / preview_every + 1) * preview_every;
            } else {
                target = starts[std::min(k, n_chunks)];
                k *= 2;
            }
            nrrt_render_stats ps;
            if (nrrt_accum_render(acc, (uint32_t)std::min<uint64_t>(target, spp), &ps) != NRRT_OK) die(nrrt_last_error(ctx));
            st.paths += ps.paths, st.segments += ps.segments, st.launches += ps.launches, st.device_ms += ps.device_ms;
            const uint32_t done = nrrt_accum_samples(acc);
            const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            if (verbose && adaptive)
                std::fprintf(stderr, "pass: %u / %u samples  %u pixels rendered  %u active  %llu segments  (%.3f s)\n", done,
                             spp, ps.pixels, nrrt_accum_active(acc), (unsigned long long)ps.segments, secs);
            else if (verbose)
                std::fprintf(stderr, "pass: %u / %u samples  (%.3f s)\n", done, spp, secs);
            if (preview_every && more()) {
                if (nrrt_accum_image(acc, image.data(), 0) != NRRT_OK ||
                    nrrt_encode_rgb8(ctx, image.data(), cam.width, cam.height, gamma, 0, preview.data()) != NRRT_OK)
                    die(nrrt_last_error(ctx));
                replace_image(output, png, preview.data(), cam.width, cam.height);
            }
        }
        if (nrrt_accum_image(acc, image.data(), 0) != NRRT_OK) die(nrrt_last_error(ctx));
        nrrt_accum_free(acc);
    } else if (nrrt_render(ctx, &cam, &opts, image.data(), verbose ? on_progress : nullptr, nullptr, &st) != NRRT_OK)
        die(nrrt_last_error(ctx));
    auto t1 = std::chrono::steady_clock::now();
    std::vector<uint8_t> rgb8(image.size());
    if (nrrt_encode_rgb8(ctx, image.data(), cam.width, cam.height, gamma, 0, rgb8.data()) != NRRT_OK) die(nrrt_last_error(ctx));
    if (out) {
        write_image(out, png, rgb8.data(), cam.width, cam.height);
        std::fclose(out);
    } else {
        replace_image(output, png, rgb8.data(), cam.width, cam.height);
    }
    if (verbose) {
        double s = std::chrono::duration<double>(t1 - t0).count();
        std::printf("Rendering: done in %.3f secs  (%ux%u, %u spp, depth %u; %llu paths, %llu ray segments, %.1f Mrays/s)\n",
                    s, cam.width, cam.height, cam.samples_per_pixel, cam.ray_max_bounces, (unsigned long long)st.paths,
                    (unsigned long long)st.segments, st.segments / (st.device_ms * 1e3));
        std::printf("Exporting: %s\n", output.c_str());
    }
    nrrt_destroy(ctx);
    nrrt_host_free(hs);
    nrrt_loaded_free(ls);
    return 0;
}
