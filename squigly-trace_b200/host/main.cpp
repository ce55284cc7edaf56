// main.cpp -- the squigly-trace command line (app/Main.hs:13-75) driving the B200 backend.
// Flags follow the cmdargs record of the reference: -s/--samples, -d/--dimensions W,H, -p/--savepath,
// --objpath, -c/--camerapath, --debug, --debugpath, --cast ; plus --bounces, --gpus, --corrected, --seed, --progress,
// --adaptive, --denoise, --aa, --lens.
#include <cctype>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <iostream>
#include <vector>

#include "squigly.hpp"

using namespace squigly;

static void usage() {
    std::cout << "squigly-trace was made by Ruko (https://github.com/rukokarasu/)  [B200 backend]\n\n"
                 "squigly [OPTIONS]\n  A cute raytracer\n\nCommon flags:\n"
                 "  -s --samples=INT       How many samples per pixel to trace\n"
                 "  -d --dimensions=INT,INT Dimensions of the resulting image\n"
                 "  -p --savepath=FILE     Where to save the output\n"
                 "     --objpath=FILE      File to load .obj from\n"
                 "  -c --camerapath=FILE   File to load camera data from\n"
                 "     --debug             Run in debug mode\n"
                 "     --debugpath=FILE    File to write debug info to\n"
                 "     --cast              Raycast instead of raytracing (i.e. don't bounce rays)\n"
                 "     --bounces=INT       Intersections per path (reference: 3)\n"
                 "     --gpus=INT          Number of B200s to use\n"
                 "     --corrected         Width x height image with per-axis offsets (default: Lib.hs index convention)\n"
                 "     --seed=INT          RNG key\n"
                 "     --progress=INT      Render in chunks of INT samples, saving a preview after each\n"
                 "     --adaptive=REL[,ABS[,MIN]]  With --progress: after each chunk stop sampling the pixels whose\n"
                 "                         standard error is below max(REL * mean, ABS) (after at least MIN samples, default 16)\n"
                 "     --denoise[=LEVELS]  With --progress: also save <savepath stem>-denoised.png after each chunk, filtered\n"
                 "                         with LEVELS (0..8, default 5) levels of the edge-aware denoiser\n"
                 "     --aa                Anti-aliasing: jitter every sample over its pixel (box filter)\n"
                 "     --lens=APERTURE,FOCUS  Depth of field: thin lens of radius APERTURE (>= 0) focused at ray parameter\n"
                 "                         FOCUS (> 0) along the camera ray\n"
                 "  -? --help              Display help message\n";
}

static std::string showTime() {      // formatTime defaultTimeLocale "%T%P UTC"
    std::time_t t = std::time(nullptr);
    char buf[64];
    std::strftime(buf, sizeof buf, "%T%P UTC", std::gmtime(&t));
    return buf;
}

// --lens=APERTURE,FOCUS: a finite aperture >= 0 and a finite focus distance > 0
static void parseLens(const std::string &v, Settings &st) {
    const std::runtime_error bad("Could not parse --lens=" + v + ", expected APERTURE,FOCUS with a number APERTURE >= 0 and a number FOCUS > 0");
    const size_t c = v.find(',');
    if (c == std::string::npos) throw bad;
    auto num = [&](const std::string &s) {
        if (s.empty() || !(std::isdigit((unsigned char)s[0]) || s[0] == '.')) throw bad;
        char *e = nullptr;
        const double d = std::strtod(s.c_str(), &e);
        if (*e || !std::isfinite(d) || !std::isfinite((float)d)) throw bad;
        return (float)d;
    };
    st.aperture = num(v.substr(0, c));
    st.focus = num(v.substr(c + 1));
    if (!(st.focus > 0.0f)) throw bad;
}

// --adaptive=REL[,ABS[,MIN]]: finite non-negative tolerances, MIN an integer >= 2
static void parseAdaptive(const std::string &v, Settings &st) {
    const std::runtime_error bad("Could not parse --adaptive=" + v + ", expected REL[,ABS[,MIN]] with non-negative numbers REL, ABS and an integer MIN >= 2");
    std::vector<std::string> f;
    for (size_t b = 0;;) {
        const size_t c = v.find(',', b);
        f.push_back(v.substr(b, c == std::string::npos ? std::string::npos : c - b));
        if (c == std::string::npos) break;
        b = c + 1;
    }
    if (f.size() > 3) throw bad;
    for (const std::string &s : f)
        if (s.empty() || !(std::isdigit((unsigned char)s[0]) || s[0] == '.')) throw bad;
    auto tol = [&](const std::string &s) {
        char *e = nullptr;
        const double d = std::strtod(s.c_str(), &e);
        if (*e || !std::isfinite(d) || d < 0.0 || !std::isfinite((float)d)) throw bad;
        return (float)d;
    };
    st.adaptiveRel = tol(f[0]);
    if (f.size() > 1) st.adaptiveAbs = tol(f[1]);
    if (f.size() > 2) {
        char *e = nullptr;
        const long long m = std::strtoll(f[2].c_str(), &e, 10);
        if (*e || m < 2 || m > INT_MAX) throw bad;
        st.adaptiveMin = (int)m;
    }
    st.adaptive = true;
}

int main(int argc, char **argv) {
    Settings st;
    try {
        for (int i = 1; i < argc; ++i) {
            std::string a = argv[i], val;
            auto eq = a.find('=');
            bool has_val = false;
            if (a.rfind("--", 0) == 0 && eq != std::string::npos) { val = a.substr(eq + 1); a = a.substr(0, eq); has_val = true; }
            auto need = [&]() -> std::string {
                if (has_val) return val;
                if (i + 1 >= argc) throw std::runtime_error("Missing value for flag " + a);
                return argv[++i];
            };
            if (a == "-s" || a == "--samples") st.samples = std::stoi(need());
            else if (a == "-d" || a == "--dimensions") {
                const std::string d = need(); const auto c = d.find(',');
                if (c == std::string::npos) throw std::runtime_error("Could not parse dimensions, expected INT,INT");
                st.dimensions = {std::stoi(d.substr(0, c)), std::stoi(d.substr(c + 1))};
            } else if (a == "-p" || a == "--savepath") st.savePath = need();
            else if (a == "--objpath") st.objPath = need();
            else if (a == "-c" || a == "--camerapath") st.cameraPath = need();
            else if (a == "--debug") st.debug = true;
            else if (a == "--debugpath") st.debugPath = need();
            else if (a == "--cast") st.cast = true;
            else if (a == "--bounces") st.bounces = std::stoi(need());
            else if (a == "--gpus") st.gpus = std::stoi(need());
            else if (a == "--corrected") st.corrected = true;
            else if (a == "--seed") st.seed = std::stoull(need());
            else if (a == "--progress") { st.progress = std::stoi(need()); if (st.progress < 1) throw std::runtime_error("--progress must be at least 1"); }
            else if (a == "--adaptive") parseAdaptive(need(), st);
            else if (a == "--denoise") {
                st.denoise = 5;
                if (has_val) {
                    if (val.empty() || val.size() > 1 || !std::isdigit((unsigned char)val[0]) || val[0] > '8')
                        throw std::runtime_error("Could not parse --denoise=" + val + ", expected LEVELS in 0..8");
                    st.denoise = val[0] - '0';
                }
            }
            else if (a == "--aa") st.aa = true;
            else if (a == "--lens") parseLens(need(), st);
            else if (a == "-?" || a == "--help") { usage(); return 0; }
            else throw std::runtime_error("Unknown flag: " + a);
        }
        if (st.adaptive && st.progress < 1) throw std::runtime_error("--adaptive needs --progress=N");
        if (st.denoise >= 0 && st.progress < 1) throw std::runtime_error("--denoise needs --progress=N");
        if (st.denoise >= 0 && (st.aa || st.focus > 0.0f))
            throw std::runtime_error("--denoise cannot be combined with --aa or --lens: the denoiser needs the primary hits, which such frames do not trace");
        if (st.cast && (st.aa || st.focus > 0.0f)) throw std::runtime_error("--cast cannot be combined with --aa or --lens");
        // main (Main.hs:35-47)
        const Camera cam = loadCamera(st.cameraPath);
        // loadBIH (Main.hs:63-75)
        ParsedScene tris = trisFromObj(st.debug, readFile(st.objPath));
        const BIH bih = makeBIH(std::move(tris));
        if (st.debug) {
            FILE *f = std::fopen(st.debugPath.c_str(), "w");
            if (!f) throw std::runtime_error(st.debugPath + ": openFile: does not exist (No such file or directory)");
            const std::string s = showBIH(bih); std::fwrite(s.data(), 1, s.size(), f); std::fclose(f);
            std::cout << "Wrote BIH to " << st.debugPath << "\n";
            std::cout << "BIH height is " << height(bih) << "\n";
            std::cout << "Length of longest leaf is " << longestLeaf(bih) << "\n";
            std::cout << "Number of leaves is " << numLeaves(bih) << "\n";
        }
        const SceneBIH scene = sceneFromBIH(bih, st.gpus);
        std::cout << "Rendering scene...\n";
        const auto t0 = std::chrono::steady_clock::now();
        std::cout << "Started at " << showTime() << "\n";
        const RenderReport rep = render(scene, cam, st);
        const auto t1 = std::chrono::steady_clock::now();
        std::cout << "Finished at " << showTime() << "\n";
        std::cout << "Took " << std::chrono::duration<double>(t1 - t0).count() << "s\n";
        if (st.debug)
            std::cout << "device " << rep.stats.device_ms << " ms, " << rep.stats.rays_traced << " rays, " << rep.stats.samples
                      << " samples, " << (rep.stats.rays_traced / (rep.stats.device_ms * 1e3)) << " Mrays/s\n";
    } catch (const std::exception &e) {
        std::cerr << "squigly-trace: " << e.what() << "\n";
        return 1;
    }
    return 0;
}
