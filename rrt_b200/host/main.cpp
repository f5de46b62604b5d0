// main.cpp -- drop-in `rrt` / `rrtd` executable over librrtb200.so.
//
// Same command line, same stdout/stderr protocol and same exit codes as the reference's main.cpp:
//   flags            -i -o -w -h -s -d -b -tx -ty -q -D          (reference main.cpp:69-119; -h is HEIGHT)
//   additions        -S <seed>  (Philox key, default 1984 = the reference's curand seed, rrt.cu:88)
//                    -R         count ray segments in a second, untimed pass (Mrays/s in the stats line; off: 0)
//                    -I <list>  frame batch (reference README.md:64 to-do "input list of scenes to render")
//                    -G <n>     n GPUs of this box: one context + one host thread per GPU, each renders its
//                               interleaved tiles; the shards are disjoint, so summing them is exact
//                    -A <prefix> linear float PFMs after the render: <prefix>.color.pfm (sum / spp) and the first-hit
//                               AOVs <prefix>.{albedo,normal,depth,coverage}.pfm (rrtb_render_aov, on the first device)
//   usage + exit 1   on any unknown argument                       (main.cpp:33-51)
//   exit 1 "no scene loaded" / 2 cannot open / 3 unknown material / 4 missing camera|materials|objects
//                                                                  (main.cpp:126-127, scene.h:220-223,287-290,431-442)
//   stdout           PPM "P3" text when no -o                      (main.cpp:140-149, color.h:25-32)
//   -o file.png      8-bit PNG, rows top-down                      (main.cpp:150-167)
//   stderr           parser summary (scene.h:443-451), banner, "took N seconds.", and the CSV stats line
//                    (rrt.cu:198-202,302,312-315) with extra fields appended at the END only.
#include <ctime>
#include <climits>
#include <cstring>
#include <iomanip>
#include <algorithm>
#include <fstream>
#include <iostream>
#include <memory>
#include <vector>
#include <string>
#include <unistd.h>

#include "rrt.h"

static void query_cuda_info() // main.cpp:13-30 (through the C ABI; one context per visible device)
{
    for (int i = 0;; ++i) {
        rrtb_ctx *c = nullptr;
        if (rrtb_create(&c, i) != RRTB_OK) break;
        int64_t info[4];
        char name[256];
        rrtb_device_info(c, info, name, sizeof(name));
        std::cout << "cudaGetDeviceProperties #" << i << "\n";
        std::cout << "  name                        " << name << "\n";
        std::cout << "  major.minor                 " << info[3] / 10 << "." << info[3] % 10 << "\n";
        std::cout << "  multiProcessorCount         " << info[0] << "\n";
        std::cout << "  l2CacheSize                 " << info[2] << "\n";
        rrtb_destroy(c);
    }
}

static void usage(const char *argv)
{
    std::cerr << "Unexpected argument: " << argv << "\n\n";
    std::cerr << "Usage: rrt [options]\n";
    std::cerr << "  -i file.txt         : input scene file\n";
    std::cerr << "  -o file.png         : output raytraced PNG image (default is PPM to stdout)\n";
    std::cerr << "  -w <width>          : output image width. (default = 1200)\n";
    std::cerr << "  -h <height>         : output image height. (800)\n";
    std::cerr << "  -s <samples>        : number of samples per pixel. (10)\n";
    std::cerr << "  -d <max_depth>      : may ray recursion depth. (50)\n";
    std::cerr << "  -b                  : disable bvh acceleration (enabled).\n";
    std::cerr << "  -tx <num_threads_x> : number of threads per block in x. (8)\n";
    std::cerr << "  -ty <num_threads_y> : number of threads per block in y. (8)\n";
    std::cerr << "  -q                  : query devices & cuda info\n";
    std::cerr << "  -D <device number>  : use this cuda device (0)\n";
    std::cerr << "  -S <seed>           : random seed (1984)\n";
    std::cerr << "  -R                  : count ray segments in a second untimed pass (rays, Mrays/s in the stats line)\n";
    std::cerr << "  -G <n>              : render on n GPUs (devices D..D+n-1), interleaved 8x4-pixel tiles (1)\n";
    std::cerr << "  -I list.txt         : frame batch: one '<scene.txt> <out.png>' per line; scenes that differ only\n";
    std::cerr << "                        in their camera reuse the uploaded scene and its BVH\n";
    std::cerr << "  -A <prefix>         : also write <prefix>.color.pfm (linear mean) and the first-hit AOVs\n";
    std::cerr << "                        <prefix>.albedo.pfm, .normal.pfm, .depth.pfm, .coverage.pfm (not with -I)\n";
    std::exit(1);
}

// same primitives and materials (camera may differ)?
static bool same_geometry(const rrtb_scene *a, const rrtb_scene *b)
{
    int32_t ca[6], cb[6];
    rrtb_scene_counts(a, ca);
    rrtb_scene_counts(b, cb);
    for (int k = 0; k < 4; ++k)
        if (ca[k] != cb[k]) return false;
    const int nmt = rrtb_scene_mtriangle_count(a);
    if (nmt != rrtb_scene_mtriangle_count(b)) return false;
    const rrtb_camera *cam_a = rrtb_scene_camera(a), *cam_b = rrtb_scene_camera(b);
    // boxes of moving spheres / moving triangles span the shutter
    if (ca[2] + nmt > 0 && (cam_a->time0 != cam_b->time0 || cam_a->time1 != cam_b->time1)) return false;
    if (nmt > 0 && memcmp(rrtb_scene_mtriangles(a), rrtb_scene_mtriangles(b), sizeof(rrtb_mtriangle) * nmt) != 0) return false;
    return memcmp(rrtb_scene_materials(a), rrtb_scene_materials(b), sizeof(rrtb_material) * ca[0]) == 0 &&
           (ca[1] == 0 || memcmp(rrtb_scene_spheres(a), rrtb_scene_spheres(b), sizeof(rrtb_sphere) * ca[1]) == 0) &&
           (ca[2] == 0 || memcmp(rrtb_scene_mspheres(a), rrtb_scene_mspheres(b), sizeof(rrtb_msphere) * ca[2]) == 0) &&
           (ca[3] == 0 || memcmp(rrtb_scene_triangles(a), rrtb_scene_triangles(b), sizeof(rrtb_triangle) * ca[3]) == 0);
}

static rrtb_scene *load_scene_or_exit(const std::string &filename, int w, int h, bool verbose)
{
    rrtb_scene *sc = nullptr;
    int code = 0;
    char err[512];
    if (rrtb_scene_parse_file(filename.c_str(), w, h, &sc, &code, err, sizeof(err)) != RRTB_OK) {
        std::cerr << err << std::endl;
        std::exit(code);
    }
    if (verbose) {
        int32_t c[6];
        rrtb_scene_counts(sc, c);
        std::cerr << "read scene file: " << filename << "\n";
        std::cerr << "material count:  " << c[0] << "\n";
        std::cerr << "sphere count:    " << c[1] << std::endl;
        std::cerr << "msphere count:   " << c[2] << std::endl;
        std::cerr << "obj count:       " << c[4] << std::endl;
        std::cerr << "obj_inst count:  " << c[5] << std::endl;
        const rrtb_camera *cam = rrtb_scene_camera(sc);
        if (cam->time0 != cam->time1) std::cerr << "camera time:     " << cam->time0 << " - " << cam->time1 << std::endl;
    }
    return sc;
}

// -I list: "<scene.txt> <out.png>" per line, one context, geometry uploaded only when it changes
static int run_batch(const std::string &list, int w, int h, int spp, int depth, bool use_bvh, int tx, int ty, int device,
                     unsigned long long seed, bool count_rays)
{
    std::ifstream fl(list);
    if (!fl.good()) {
        std::cerr << "ERROR: problem with opening file: " << list << "\n";
        return 2;
    }
    Rrt rrt(w, h, spp, depth, use_bvh, tx, ty, device, seed);
    rrt.count_rays = count_rays;
    rrtb_scene *prev = nullptr;
    std::string scene_file, png_file;
    std::vector<uint8_t> rgb((size_t)w * h * 3);
    int frames = 0, uploads = 0;
    double seconds = 0.0;
    unsigned long long rays = 0;
    while (fl >> scene_file >> png_file) {
        rrtb_scene *cur = load_scene_or_exit(scene_file, w, h, false);
        vec3 *fb;
        if (prev && same_geometry(prev, cur)) {
            fb = rrt.render_camera_only(cur);
        }
        else {
            fb = rrt.render(cur);
            ++uploads;
        }
        seconds += rrt.stats.seconds_render;
        rays += rrt.stats.rays;
        rrtb_tonemap_fp(&fb[0].e[0], w, h, spp, rgb.data());
        if (rrtb_write_png(png_file.c_str(), w, h, rgb.data()) != RRTB_OK) {
            std::cerr << "ERROR: could not write " << png_file << std::endl;
            return 1;
        }
        if (prev) rrtb_scene_free(prev);
        prev = cur;
        ++frames;
    }
    if (prev) rrtb_scene_free(prev);
    std::cerr << "batch: " << frames << " frames, " << uploads << " scene uploads, " << seconds << " render seconds, "
              << (seconds > 0 ? rays / seconds * 1e-6 : 0.0) << " Mrays/s\n";
    return 0;
}

int main(int argc, char *argv[])
{
    int image_width = 1200, image_height = 800, num_samples = 10;
    int num_threads_x = 8, num_threads_y = 8;
    std::string the_scene_filename;
    char *png_filename = nullptr;
    int max_depth = 50;
    bool use_bvh = true;
    int device = 0;
    unsigned long long seed = 1984;
    std::string batch_list;
    int n_gpus = 1;
    bool count_rays = false;
    std::string aov_prefix;

    // Only the first letter after '-' is examined, as in the reference (so "-input" == "-i").
    for (int i = 1; i < argc; ++i) {
        if (argv[i][0] != '-') usage(argv[i]);
        const char c = argv[i][1];
        auto next = [&]() -> char * {
            if (i + 1 >= argc) usage(argv[i]);
            return argv[++i];
        };
        if (c == 'i') the_scene_filename = next();
        else if (c == 'o') png_filename = next();
        else if (c == 'w') image_width = atoi(next());
        else if (c == 'h') image_height = atoi(next());
        else if (c == 's') num_samples = atoi(next());
        else if (c == 'd') max_depth = atoi(next());
        else if (c == 'b') use_bvh = false;
        else if (c == 't') {
            if (argv[i][2] == 'x') num_threads_x = atoi(next());
            else if (argv[i][2] == 'y') num_threads_y = atoi(next());
            else usage(argv[i]);
        }
        else if (c == 'q') query_cuda_info();
        else if (c == 'D') device = atoi(next());
        else if (c == 'S') seed = strtoull(next(), nullptr, 10);
        else if (c == 'I') batch_list = next();
        else if (c == 'G') n_gpus = atoi(next());
        else if (c == 'R') count_rays = true;
        else if (c == 'A') aov_prefix = next();
        else usage(argv[i]);
    }
    if (aov_prefix != "" && batch_list != "") usage("-A (with -I)");

    if (batch_list != "")
        return run_batch(batch_list, image_width, image_height, num_samples, max_depth, use_bvh, num_threads_x, num_threads_y,
                         device, seed, count_rays);

    rrtb_scene *the_scene = nullptr;
    if (the_scene_filename != "") {
        int code = 0;
        char err[512];
        if (rrtb_scene_parse_file(the_scene_filename.c_str(), image_width, image_height, &the_scene, &code, err,
                                  sizeof(err)) != RRTB_OK) {
            std::cerr << err << std::endl;
            std::exit(code);
        }
        int32_t c[6];
        rrtb_scene_counts(the_scene, c);
        std::cerr << "read scene file: " << the_scene_filename << "\n";
        std::cerr << "material count:  " << c[0] << "\n";
        std::cerr << "sphere count:    " << c[1] << std::endl;
        std::cerr << "msphere count:   " << c[2] << std::endl;
        std::cerr << "obj count:       " << c[4] << std::endl;
        std::cerr << "obj_inst count:  " << c[5] << std::endl;
        const rrtb_camera *cam = rrtb_scene_camera(the_scene);
        if (cam->time0 != cam->time1) std::cerr << "camera time:     " << cam->time0 << " - " << cam->time1 << std::endl;
    }
    else {
        std::cerr << "ERROR: no scene loaded." << std::endl;
        std::exit(1);
    }

    std::time_t render_time = std::time(nullptr);
    std::tm render_tm = *std::localtime(&render_time);

    // -G n: n contexts, one per device D..D+n-1 (RRTB_GROUP_SAME_DEVICE=1: all on device D, a test aid for boxes with
    // one GPU); ONE library call renders all shards and combines them over NVLink (rrtb_render_group)
    if (n_gpus < 1) n_gpus = 1;
    const bool same_device = getenv("RRTB_GROUP_SAME_DEVICE") != nullptr;
    Rrt rrt(image_width, image_height, num_samples, max_depth, use_bvh, num_threads_x, num_threads_y, device, seed);
    rrt.count_rays = count_rays;
    std::vector<std::unique_ptr<Rrt>> peers;
    for (int r = 1; r < n_gpus; ++r)
        peers.emplace_back(new Rrt(image_width, image_height, num_samples, max_depth, use_bvh, num_threads_x, num_threads_y,
                                   same_device ? device : device + r, seed));
    std::cerr << "Rendering a " << image_width << "x" << image_height << " image with " << num_samples
              << " samples per pixel on a persistent sm_100a kernel.\n";
    int32_t c[6];
    rrtb_scene_counts(the_scene, c);
    std::cerr << "num_hittables = " << (c[1] + c[2] + c[3]) << "\n";
    std::cerr << "CUDA Device: " << device << std::endl;

    vec3 *fb;
    if (n_gpus == 1) {
        fb = rrt.render(the_scene);
    }
    else {
        std::vector<Rrt *> others;
        for (auto &q : peers) others.push_back(q.get());
        fb = rrt.render_group(the_scene, others);
    }

    const double timer_seconds = rrt.stats.seconds_render;
    std::cerr << "took " << timer_seconds << " seconds.\n";
    char hostname[HOST_NAME_MAX + 1];
    gethostname(hostname, sizeof(hostname));
    // reference fields first (rrt.cu:312-315): date,host,CUDA<ver>,FP_T,W,H,spp,blocks,tx,ty,seconds ; then ours
    std::cerr << "stats," << std::put_time(&render_tm, "%c %Z,") << std::string(hostname) << ","
              << "CUDA-rrtb" << rrtb_abi_version() << "," RRTB_FP_NAME "," << image_width << "," << image_height << ","
              << num_samples << "," << rrt.stats.kernel_launches << "," << num_threads_x << "," << num_threads_y << ","
              << timer_seconds << "," << rrt.stats.rays << ","
              << (timer_seconds > 0 ? rrt.stats.rays / timer_seconds * 1e-6 : 0.0) << "," << rrt.stats.seconds_build
              << "," << (n_gpus < 1 ? 1 : n_gpus) << "\n";

    if (png_filename == nullptr) {
        // PPM to stdout: rows top-down, one "r g b" line per pixel (main.cpp:140-149)
        std::vector<uint8_t> rgb((size_t)image_width * image_height * 3);
        rrtb_tonemap_fp(&fb[0].e[0], image_width, image_height, num_samples, rgb.data());
        std::cout << "P3\n" << image_width << ' ' << image_height << "\n255\n";
        for (size_t k = 0; k < rgb.size(); k += 3)
            std::cout << (int)rgb[k] << ' ' << (int)rgb[k + 1] << ' ' << (int)rgb[k + 2] << '\n';
    }
    else {
        std::vector<uint8_t> rgb((size_t)image_width * image_height * 3);
        rrtb_tonemap_fp(&fb[0].e[0], image_width, image_height, num_samples, rgb.data());
        if (rrtb_write_png(png_filename, image_width, image_height, rgb.data()) != RRTB_OK) {
            std::cerr << "ERROR: could not write " << png_filename << std::endl;
            std::exit(1);
        }
    }
    if (aov_prefix != "") { // linear PFMs: the beauty mean, then the first-hit AOVs at the same samples, seed and precision
        const size_t n = (size_t)image_width * image_height;
        std::vector<float> color(3 * n), albedo(3 * n), normal(3 * n), depth(n), coverage(n);
        for (size_t k = 0; k < n; ++k)
            for (int c = 0; c < 3; ++c) color[3 * k + c] = (float)(fb[k].e[c] / (FP_T)num_samples);
        rrt.render_aov(albedo.data(), normal.data(), depth.data(), coverage.data());
        const struct {
            const char *name;
            int channels;
            const float *data;
        } pfm[5] = {{".color.pfm", 3, color.data()}, {".albedo.pfm", 3, albedo.data()}, {".normal.pfm", 3, normal.data()},
                    {".depth.pfm", 1, depth.data()}, {".coverage.pfm", 1, coverage.data()}};
        for (const auto &f : pfm) {
            const std::string path = aov_prefix + f.name;
            if (rrtb_write_pfm(path.c_str(), image_width, image_height, f.channels, f.data) != RRTB_OK) {
                std::cerr << "ERROR: could not write " << path << std::endl;
                std::exit(1);
            }
        }
    }
    rrtb_scene_free(the_scene);
    return 0;
}
