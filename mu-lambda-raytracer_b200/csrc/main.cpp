// rt_main — the command-line host of the reference (src/main.rs) over the C ABI of librt_b200.
//
// Same flags, defaults and output as the reference binary:
//   --aspect_ratio W:H (16:9)  --image_width N (400)  --samples_per_pixel N (200)  --max_depth N (50)
//   --lookfrom x,y,z  --lookat x,y,z  --up x,y,z (0,1.0,0)  --field_of_view DEG  --aperture A (0.0)  --focus_dist D
//   --world NAME (simple)  --seed N  --randomized_rendering | -r                        main.rs:64-132
//   stdout: "P3\nW H\n255\n" then one "r g b" line per pixel, top row first             main.rs:144,175-179
//   stderr: "Remaining: NN%" progress, "Done!", "Rendered in X.XXXs"                    main.rs:157-174
// Both `--flag=value` and `--flag value` are accepted, like clap 2.  Usage errors exit with 1 (clap), values that the
// reference would `unwrap()` into a panic exit with 101 (Rust's panic exit code).
// Additions that do not exist in the reference: --gpus N (devices of this box to shard over), --pipeline NAME,
// --earthmap FILE (decoded RGB8 as binary PPM; default $RT_EARTHMAP, ./earthmap.ppm, then the shipped asset),
// --stats (one JSON line with paths, rays, device ms on stderr), --noise_threshold T with --min_samples N (16): adaptive
// sampling, every pixel until the standard error of its displayed value is at most T, --samples_per_pixel at most
// (rt_render_adaptive; T = 0, the default, renders the fixed count; one GPU only), --denoise: the variance-guided
// non-local-means filter with the library's default parameters after the render, uniform or adaptive (rt_render_denoised;
// one GPU only; --stats then covers the render and the filter), --denoise_guided: the same with the feature-guided filter
// and its default parameters (rt_render_denoised_guided; implies --denoise; --stats also covers the feature pass),
// --denoise_dual: dual-buffer cross filtering (rt_render_denoised_dual; implies --denoise, combines with --denoise_guided,
// and with --noise_threshold the stop rule judges the filtered value; --samples_per_pixel and --min_samples must be even),
// --denoise_sure: per-pixel selection among three strengths of the cross filter by a risk estimate, which also drives the stop
// rule with --noise_threshold (rt_render_denoised_sure with the library's default RtSure; implies --denoise_dual),
// --noise_prior: the stop rule of --noise_threshold with each pixel's variance pooled with its neighbourhood's (the library's
// default RtPrior: rt_render_adaptive_prior, or rt_render_denoised_sure_prior with --denoise_sure; needs --noise_threshold, and
// of the filters only --denoise_sure).
// There is no CPU renderer here: without a CUDA device the program fails with the library's error.
#include <unistd.h>

#include <cctype>
#include <cerrno>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <random>
#include <string>
#include <vector>

#include "../../include/rt_b200.h"

namespace {

[[noreturn]] void usage_error(const std::string& msg) {  // clap::Error::exit
    fprintf(stderr, "error: %s\n\nUSAGE:\n    rt_main [OPTIONS]\n\nFor more information try --help\n", msg.c_str());
    exit(1);
}
[[noreturn]] void panic(const std::string& msg) {  // .unwrap() on a bad value
    fprintf(stderr, "thread 'main' panicked: %s\n", msg.c_str());
    exit(101);
}

long long parse_int(const std::string& s, const char* what) {
    char* end = nullptr;
    errno = 0;
    long long v = strtoll(s.c_str(), &end, 10);
    if (s.empty() || *end || errno) panic(std::string("invalid integer for ") + what + ": '" + s + "'");
    return v;
}
uint64_t parse_u64(const std::string& s, const char* what) {
    char* end = nullptr;
    errno = 0;
    if (s.empty() || s[0] == '-') panic(std::string("invalid u64 for ") + what + ": '" + s + "'");
    unsigned long long v = strtoull(s.c_str(), &end, 10);
    if (*end || errno) panic(std::string("invalid u64 for ") + what + ": '" + s + "'");
    return v;
}
double parse_f64(const std::string& s, const char* what) {
    char* end = nullptr;
    double v = strtod(s.c_str(), &end);
    if (s.empty() || *end) panic(std::string("invalid float for ") + what + ": '" + s + "'");
    return v;
}
double parse_aspect_ratio(const std::string& s) {  // main.rs:49-52: i32 / i32 as f64
    size_t c = s.find(':');
    if (c == std::string::npos) panic("aspect_ratio must be W:H");
    return (double)(int32_t)parse_int(s.substr(0, c), "aspect_ratio") / (double)(int32_t)parse_int(s.substr(c + 1), "aspect_ratio");
}
void parse_vector(const std::string& s, double out[3], const char* what) {  // main.rs:54-62
    size_t pos = 0;
    for (int i = 0; i < 3; ++i) {
        size_t c = s.find(',', pos);
        if (i < 2 && c == std::string::npos) panic(std::string(what) + " must be x,y,z");
        out[i] = parse_f64(s.substr(pos, c == std::string::npos ? std::string::npos : c - pos), what);
        pos = c + 1;
    }
}

bool read_ppm(const std::string& path, std::vector<uint8_t>& rgb, int& w, int& h) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    std::vector<uint8_t> data;
    uint8_t buf[1 << 16];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, f)) > 0) data.insert(data.end(), buf, buf + n);
    fclose(f);
    if (data.size() < 2 || data[0] != 'P' || data[1] != '6') return false;
    size_t pos = 2;
    long fields[3];
    for (int k = 0; k < 3; ++k) {
        for (;;) {
            while (pos < data.size() && isspace(data[pos])) ++pos;
            if (pos < data.size() && data[pos] == '#') {
                while (pos < data.size() && data[pos] != '\n') ++pos;
                continue;
            }
            break;
        }
        long v = 0;
        bool any = false;
        while (pos < data.size() && isdigit(data[pos])) v = v * 10 + (data[pos++] - '0'), any = true;
        if (!any) return false;
        fields[k] = v;
    }
    pos += 1;  // the single whitespace byte after maxval
    w = (int)fields[0], h = (int)fields[1];
    if (fields[2] != 255 || w <= 0 || h <= 0 || data.size() < pos + (size_t)3 * w * h) return false;
    rgb.assign(data.begin() + pos, data.begin() + pos + (size_t)3 * w * h);
    return true;
}

std::string exe_dir(const char* argv0) {
    char buf[4096];
    ssize_t n = readlink("/proc/self/exe", buf, sizeof buf - 1);
    std::string p = n > 0 ? std::string(buf, (size_t)n) : std::string(argv0);
    size_t s = p.rfind('/');
    return s == std::string::npos ? "." : p.substr(0, s);
}

struct Progress {  // the logger closure of do_tracing (main.rs:157-173): called once per row, counts the rows down
    std::chrono::steady_clock::time_point start;
    long long last_logged_ms = 0;
    int remaining = -1;
};
void progress_cb(int /*row*/, int total, void* user) {
    Progress* p = (Progress*)user;
    if (p->remaining < 0) p->remaining = total;
    p->remaining -= 1;
    if (p->remaining == 0) {
        fprintf(stderr, "\r%-50s", "Done!");
        return;
    }
    long long elapsed = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - p->start).count();
    if (elapsed - p->last_logged_ms > 300) {
        p->last_logged_ms = elapsed;
        fprintf(stderr, "\rRemaining: %3d%%  ", (int)((long long)p->remaining * 100 / total));
    }
}

}  // namespace

int main(int argc, char** argv) {
    // ---- flags (main.rs:64-88)
    std::map<std::string, std::string> defaults = {{"aspect_ratio", "16:9"}, {"image_width", "400"}, {"samples_per_pixel", "200"},
                                                   {"max_depth", "50"},      {"up", "0,1.0,0"},     {"aperture", "0.0"},
                                                   {"world", "simple"},      {"gpus", "1"},         {"pipeline", "auto"},
                                                   {"noise_threshold", "0"}, {"min_samples", "16"}};
    const char* valued[] = {"aspect_ratio", "image_width", "samples_per_pixel", "max_depth", "lookfrom", "lookat", "up", "field_of_view",
                            "aperture",     "focus_dist",  "world",             "seed",      "gpus",     "pipeline", "earthmap",
                            "noise_threshold", "min_samples"};
    std::map<std::string, std::string> opt = defaults;
    bool randomized_rendering = false, want_stats = false, want_denoise = false, want_guided = false, want_dual = false, want_sure = false,
         want_prior = false;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        if (a == "--randomized_rendering" || a == "-r") {
            randomized_rendering = true;
            continue;
        }
        if (a == "--stats") {
            want_stats = true;
            continue;
        }
        if (a == "--denoise") {
            want_denoise = true;
            continue;
        }
        if (a == "--denoise_guided") {
            want_denoise = want_guided = true;
            continue;
        }
        if (a == "--denoise_dual") {
            want_denoise = want_dual = true;
            continue;
        }
        if (a == "--denoise_sure") {
            want_denoise = want_dual = want_sure = true;
            continue;
        }
        if (a == "--noise_prior") {
            want_prior = true;
            continue;
        }
        if (a == "--help" || a == "-h") {
            printf("mulambda raytracer 0.1 (B200)\n\nUSAGE:\n    rt_main [FLAGS] [OPTIONS]\n\nFLAGS:\n    -r, --randomized_rendering\n        --stats\n        --denoise\n        --denoise_guided\n        --denoise_dual\n        --denoise_sure\n        --noise_prior\n\nOPTIONS:\n");
            for (const char* v : valued) {
                auto d = defaults.find(v);
                printf("        --%s <%s>%s%s%s\n", v, v, d != defaults.end() ? " [default: " : "", d != defaults.end() ? d->second.c_str() : "",
                       d != defaults.end() ? "]" : "");
            }
            printf("\nworlds:");
            for (int k = 0; k < rt_world_count(); ++k) printf(" %s", rt_world_name(k));
            printf("\n");
            return 0;
        }
        if (a == "--version" || a == "-V") {
            printf("mulambda raytracer 0.1\n");
            return 0;
        }
        if (a.rfind("--", 0) != 0) usage_error("Found argument '" + a + "' which wasn't expected, or isn't valid in this context");
        std::string name = a.substr(2), value;
        size_t eq = name.find('=');
        bool has_value = eq != std::string::npos;
        if (has_value) value = name.substr(eq + 1), name = name.substr(0, eq);
        bool known = false;
        for (const char* v : valued) known = known || name == v;
        if (!known) usage_error("Found argument '--" + name + "' which wasn't expected, or isn't valid in this context");
        if (!has_value) {
            if (i + 1 >= argc) usage_error("The argument '--" + name + " <" + name + ">' requires a value but none was supplied");
            value = argv[++i];
        }
        opt[name] = value;
    }

    // ---- world lookup (possible_values of --world, main.rs:79-84)
    RtWorldInfo info;
    if (rt_world_info(opt["world"].c_str(), &info) != RT_OK) {
        std::string names;
        for (int k = 0; k < rt_world_count(); ++k) names += std::string(k ? ", " : "") + rt_world_name(k);
        usage_error("'" + opt["world"] + "' isn't a valid value for '--world <world>'\n\t[possible values: " + names + "]");
    }

    // ---- parameters (main.rs:101-131)
    double aspect_ratio = parse_aspect_ratio(opt["aspect_ratio"]);
    long long image_width = parse_int(opt["image_width"], "image_width");
    if (image_width < 0) panic("image_width must be a usize");
    long long image_height = (long long)((double)image_width / aspect_ratio);  // `as usize` truncates
    long long spp = (int32_t)parse_int(opt["samples_per_pixel"], "samples_per_pixel");
    long long max_depth = (int32_t)parse_int(opt["max_depth"], "max_depth");
    RtCamera cam;
    cam.time0 = cam.time1 = 0.0;  // the reference's camera has no shutter (motion blur is an extension of the library)
    memcpy(cam.lookfrom, info.lookfrom, sizeof cam.lookfrom);
    memcpy(cam.lookat, info.lookat, sizeof cam.lookat);
    if (opt.count("lookfrom")) parse_vector(opt["lookfrom"], cam.lookfrom, "lookfrom");
    if (opt.count("lookat")) parse_vector(opt["lookat"], cam.lookat, "lookat");
    parse_vector(opt["up"], cam.vup, "up");
    cam.vfov_deg = opt.count("field_of_view") ? parse_f64(opt["field_of_view"], "field_of_view") : info.vfov_deg;
    cam.aspect_ratio = aspect_ratio;  // the flag ratio, not W/H (main.rs:197)
    cam.aperture = parse_f64(opt["aperture"], "aperture");
    if (opt.count("focus_dist")) {
        cam.focus_dist = parse_f64(opt["focus_dist"], "focus_dist");
    } else {  // (lookat - lookfrom).length()
        double d[3] = {cam.lookat[0] - cam.lookfrom[0], cam.lookat[1] - cam.lookfrom[1], cam.lookat[2] - cam.lookfrom[2]};
        cam.focus_dist = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    }
    // --seed absent: thread_rng() for the world and the pixels (main.rs:212-214); here: a fresh seed from the OS
    std::random_device rd;
    uint64_t os_seed = ((uint64_t)rd() << 32) ^ (uint64_t)rd();
    uint64_t world_seed = opt.count("seed") ? parse_u64(opt["seed"], "seed") : os_seed;
    uint64_t render_seed = (opt.count("seed") && !randomized_rendering) ? world_seed : (((uint64_t)rd() << 32) ^ (uint64_t)rd());
    long long gpus = parse_int(opt["gpus"], "gpus");
    const double noise_threshold = parse_f64(opt["noise_threshold"], "noise_threshold");
    const long long min_samples = parse_int(opt["min_samples"], "min_samples");
    if (want_prior && noise_threshold == 0.0) usage_error("--noise_prior is a prior of the stop rule: it needs --noise_threshold");
    if (want_prior && gpus > 1) usage_error("--noise_prior (adaptive sampling) renders on one GPU: it cannot be used with --gpus above 1");
    if (want_prior && want_denoise && !want_sure)
        usage_error(std::string("--noise_prior drives the plain or the SURE stop rule: it cannot be used with ") +
                    (want_dual ? "--denoise_dual" : want_guided ? "--denoise_guided" : "--denoise") + " unless --denoise_sure is also given");
    if (noise_threshold != 0.0 && gpus > 1) usage_error("--noise_threshold (adaptive sampling) renders on one GPU: it cannot be used with --gpus above 1");
    if (want_denoise && gpus > 1)
        usage_error(std::string(want_sure ? "--denoise_sure" : want_dual ? "--denoise_dual" : want_guided ? "--denoise_guided" : "--denoise") +
                    " renders and filters on one GPU: it cannot be used with --gpus above 1");
    if (want_dual && (spp % 2 != 0 || min_samples % 2 != 0))
        usage_error(std::string(want_sure ? "--denoise_sure" : "--denoise_dual") +
                    " splits every range of samples into two halves: --samples_per_pixel and --min_samples must be even");
    static const std::map<std::string, int> pipelines = {{"auto", RT_PIPELINE_AUTO}, {"megakernel", RT_PIPELINE_MEGAKERNEL},
                                                         {"wavefront", RT_PIPELINE_WAVEFRONT},
                                                         {"persistent", RT_PIPELINE_PERSISTENT}};
    if (!pipelines.count(opt["pipeline"])) usage_error("'" + opt["pipeline"] + "' isn't a valid value for '--pipeline <pipeline>'");

    // ---- World::build (main.rs:185-188)
    std::vector<uint8_t> earth;
    int ew = 0, eh = 0;
    if (info.needs_earthmap) {  // the reference opens earthmap.jpg relative to the CWD (worlds.rs:441) and unwraps
        std::vector<std::string> tries;
        if (opt.count("earthmap")) tries.push_back(opt["earthmap"]);
        else {
            if (getenv("RT_EARTHMAP")) tries.push_back(getenv("RT_EARTHMAP"));
            tries.push_back("earthmap.ppm");
            tries.push_back(exe_dir(argv[0]) + "/../assets/earthmap.ppm");
        }
        bool ok = false;
        for (auto& t : tries) ok = ok || read_ppm(t, earth, ew, eh);
        if (!ok) panic("cannot open the earthmap image (binary PPM): tried " + tries.front() + (tries.size() > 1 ? ", ..." : ""));
    }
    RtSceneDesc* desc = nullptr;
    if (rt_world_build(opt["world"].c_str(), world_seed, earth.empty() ? nullptr : earth.data(), ew, eh, &desc, nullptr) != RT_OK) {
        fprintf(stderr, "error: %s\n", rt_last_error());
        return 1;
    }

    // ---- do_tracing (main.rs:134-180)
    if (image_width < 2 || image_height < 2 || spp <= 0) {
        fprintf(stderr, "error: image must be at least 2x2 and samples_per_pixel positive (got %lldx%lld, %lld spp)\n", image_width, image_height, spp);
        return 1;
    }
    int n_dev = rt_device_count();
    if (gpus < 1 || gpus > std::max(n_dev, 1)) {
        fprintf(stderr, "error: --gpus %lld but %d CUDA device(s) are visible\n", gpus, n_dev);
        return 1;
    }
    std::vector<RtScene*> scenes((size_t)gpus, nullptr);
    for (int g = 0; g < gpus; ++g)
        if (rt_scene_create(desc, g, &scenes[g]) != RT_OK) {
            fprintf(stderr, "error: %s\n", rt_last_error());
            return 1;
        }
    printf("P3\n%lld %lld\n255\n", image_width, image_height);
    RtParams p;
    memset(&p, 0, sizeof p);
    p.width = (int32_t)image_width, p.height = (int32_t)image_height;
    p.samples_per_pixel = (int32_t)spp, p.max_depth = (int32_t)std::max<long long>(max_depth, 0);
    p.seed = render_seed, p.pipeline = pipelines.at(opt["pipeline"]), p.device = -1;
    std::vector<int32_t> rgb((size_t)3 * image_width * image_height);
    Progress prog{std::chrono::steady_clock::now(), 0};
    RtStats st;
    int rc;
    RtAdaptive ad;
    memset(&ad, 0, sizeof ad);
    ad.noise_threshold = noise_threshold, ad.min_samples = (int32_t)min_samples;
    RtPrior pr;
    memset(&pr, 0, sizeof pr);
    pr.prior_samples = RT_PRIOR_DEFAULT_SAMPLES, pr.radius = RT_PRIOR_DEFAULT_RADIUS;
    if (want_denoise) {
        RtDenoise dn;
        memset(&dn, 0, sizeof dn);
        dn.k = RT_DENOISE_DEFAULT_K, dn.alpha = RT_DENOISE_DEFAULT_ALPHA;
        dn.search_radius = RT_DENOISE_DEFAULT_SEARCH_RADIUS, dn.patch_radius = RT_DENOISE_DEFAULT_PATCH_RADIUS;
        RtGuide gd;
        memset(&gd, 0, sizeof gd);
        gd.k_feature = RT_GUIDE_DEFAULT_K_FEATURE, gd.tau = RT_GUIDE_DEFAULT_TAU, gd.feature_samples = RT_GUIDE_DEFAULT_FEATURE_SAMPLES;
        RtSure su;
        memset(&su, 0, sizeof su);
        su.ratio = RT_SURE_DEFAULT_RATIO, su.smooth_radius = RT_SURE_DEFAULT_SMOOTH_RADIUS;
        if (want_sure && want_prior) {
            rc = rt_render_denoised_sure_prior(scenes[0], &cam, &p, &ad, &dn, want_guided ? &gd : nullptr, &su, &pr, rgb.data(), nullptr, nullptr,
                                               nullptr, nullptr, progress_cb, &prog, &st);
        } else if (want_sure) {
            rc = rt_render_denoised_sure(scenes[0], &cam, &p, noise_threshold != 0.0 ? &ad : nullptr, &dn, want_guided ? &gd : nullptr, &su, rgb.data(),
                                         nullptr, nullptr, nullptr, nullptr, progress_cb, &prog, &st);
        } else if (want_dual) {
            rc = rt_render_denoised_dual(scenes[0], &cam, &p, noise_threshold != 0.0 ? &ad : nullptr, &dn, want_guided ? &gd : nullptr, rgb.data(), nullptr,
                                         nullptr, nullptr, progress_cb, &prog, &st);
        } else if (want_guided) {
            rc = rt_render_denoised_guided(scenes[0], &cam, &p, noise_threshold != 0.0 ? &ad : nullptr, &dn, &gd, rgb.data(), nullptr, progress_cb, &prog,
                                           &st);
        } else {
            rc = rt_render_denoised(scenes[0], &cam, &p, noise_threshold != 0.0 ? &ad : nullptr, &dn, rgb.data(), nullptr, progress_cb, &prog, &st);
        }
    } else if (want_prior) {
        rc = rt_render_adaptive_prior(scenes[0], &cam, &p, &ad, &pr, rgb.data(), nullptr, nullptr, nullptr, progress_cb, &prog, &st);
    } else if (noise_threshold != 0.0) {
        rc = rt_render_adaptive(scenes[0], &cam, &p, &ad, rgb.data(), nullptr, nullptr, nullptr, progress_cb, &prog, &st);
    } else {
        rc = rt_render_multi(scenes.data(), (int32_t)gpus, &cam, &p, nullptr, rgb.data(), progress_cb, &prog, &st);
    }
    if (rc != RT_OK) {
        fprintf(stderr, "\nerror: %s\n", rt_last_error());
        return 1;
    }
    double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - prog.start).count();
    fprintf(stderr, "\nRendered in %.3fs\n", secs);
    if (want_stats)
        fprintf(stderr, "{\"paths\": %llu, \"rays\": %llu, \"device_ms\": %.3f, \"kernel_launches\": %d, \"pipeline\": %d, \"gpus\": %lld, \"mpaths_per_s\": %.1f, \"mean_spp\": %.3f}\n",
                (unsigned long long)st.paths, (unsigned long long)st.rays, st.device_ms, st.kernel_launches, st.pipeline_used, gpus,
                st.paths / (st.device_ms * 1e3), (double)st.paths / ((double)image_width * (double)image_height));
    // ---- PPM body: rows in reverse j (top row first), one pixel per line
    std::string out;
    out.reserve((size_t)12 * image_width * image_height);
    char line[48];
    for (long long j = image_height - 1; j >= 0; --j)
        for (long long i = 0; i < image_width; ++i) {
            const int32_t* px = &rgb[(size_t)3 * (j * image_width + i)];
            int n = snprintf(line, sizeof line, "%d %d %d\n", px[0], px[1], px[2]);
            out.append(line, (size_t)n);
        }
    fwrite(out.data(), 1, out.size(), stdout);
    for (RtScene* s : scenes) rt_scene_destroy(s);
    rt_scene_desc_free(desc);
    return 0;
}
