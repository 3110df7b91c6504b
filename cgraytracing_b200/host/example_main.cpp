// example_main.cpp — what the reference's main() (main.cpp:268-414) looks like on top of cgrt_host.hpp: build the scene
// objects on the stack, push raw Object* into a vector, call render(objs) once, tone-map and write the picture.
//
//   example_main <scene> <width> <height> <photons> <rounds> <out.ppm> [assets-dir] [gpus] [peer|nccl] [off|jitter|corner]
//   off|jitter|corner: PPM (default) or stochastic PPM with jittered / pixel-corner camera rays (RenderOptions::sppm)
//   scenes: bunny (main.cpp:293 + chessboard floor), dragon (glass dragon, BASELINE config 3), spheres (main.cpp:288-290)
//
// Prints one line: "<hitpoints> <deposits> <fnv1a-64 of the fp64 image> <mean 8-bit level>" — tests/test_gpu_host_cpp.py
// compares it with the same render driven through the Python binding. Exit code 3 = no GPU (there is no CPU fallback).
#include <cinttypes>
#include <cstdlib>
#include <cstring>

#include "cgrt_host.hpp"

using namespace cgrt_host;

int main(int argc, char **argv) {
    if (argc < 7) {
        std::fprintf(stderr, "usage: %s <bunny|dragon|spheres> <width> <height> <photons> <rounds> <out.ppm> [assets-dir] [gpus] [peer|nccl] [off|jitter|corner] [accum_mode]\n",
                     argv[0]);
        return 2;
    }
    const std::string scene = argv[1], out = argv[6], assets = argc > 7 ? argv[7] : "cgraytracing_b200/assets";
    RenderOptions opt;
    opt.width = std::atoi(argv[2]); opt.height = std::atoi(argv[3]);
    opt.num_photon = std::atoi(argv[4]); opt.num_threads = 1; opt.rounds = std::atoi(argv[5]);
    opt.num_gpus = argc > 8 ? std::atoi(argv[8]) : 1;  // > 1: rows and photon ranges split over that many GPUs of this box
    opt.peer_exchange = argc > 9 && std::string(argv[9]) == "peer";  // accumulators exchanged over peer memory instead of ncclAllReduce
    if (argc > 10) {
        const std::string mode = argv[10];
        if (mode == "jitter") opt.sppm = CGRT_SPPM_JITTER;
        else if (mode == "corner") opt.sppm = CGRT_SPPM_CORNER;
        else if (mode != "off") { std::fprintf(stderr, "unknown mode %s (off|jitter|corner)\n", mode.c_str()); return 2; }
    }
    if (argc > 11) opt.accum_mode = std::atoi(argv[11]);  // 2: fixed-point accumulators (the same image on any GPU count)
    try {
        // floor texture: Texture(tdata, Vec3(0,1,0), Vec3(-21,0,0), 42, 40, false) — main.cpp:320 with ChessBoard.png
        int tw = 0, th = 0;
        std::vector<uint8_t> texels = read_texture_asset(assets + "/ChessBoard.cgrttex", tw, th);
        Texture tex(texels.data(), tw, th, Vec3(0, 1, 0), Vec3(-21, 0, 0), 42, 40, false);
        // the five planes of main.cpp:348-353
        Plane floor_(Vec3(0.0, -20, 0), Vec3(0, 1, 0), Vec3(0.15, 0.15, 0.15), 0.0, 0.0, tex);
        Plane right(Vec3(20, 0.0, 0), Vec3(-1, 0, 0), Vec3(0.15, 0.50, 0.15));
        Plane left(Vec3(-20, 0.0, 0), Vec3(1, 0, 0), Vec3(0.50, 0.15, 0.15));
        Plane back(Vec3(0.0, 0.0, 40), Vec3(0, 0, -1), Vec3(0.15, 0.15, 0.15));
        Plane ceiling(Vec3(0.0, 20, 0), Vec3(0, -1, 0), Vec3(0.15, 0.15, 0.15));
        std::vector<Object *> objs;
        std::unique_ptr<Object> extra[3];
        if (scene == "spheres") {  // main.cpp:288-290, pushed before the planes (:356-359)
            extra[0].reset(new Sphere(Vec3(-15.0, -20.0, 60), 10, Vec3(0.3, 0.3, 0.3), 0.0, 0.0));
            extra[1].reset(new Sphere(Vec3(10.0, -20.0, 60), 7, Vec3(1.0, 1.0, 1.0), 0.8, 0.0));
            extra[2].reset(new Sphere(Vec3(10.0, -20.0, 30), 7, Vec3(1.0, 1.0, 1.0), 0.8, 0.5));
            for (auto &e : extra) objs.push_back(e.get());
        }
        objs.push_back(&floor_); objs.push_back(&right); objs.push_back(&left); objs.push_back(&back); objs.push_back(&ceiling);
        if (scene == "bunny")  // TriangleMesh("model/lowpolybunny.txt", 10, Vec3(0,-15,40), Vec3(1,1,1), 0.8, 0.5) — main.cpp:293
            extra[0].reset(new TriangleMesh(read_mesh_asset(assets + "/lowpolybunny.cgrtmesh", 10, Vec3(0, -15, 40)), Vec3(1.0, 1.0, 1.0), 0.8, 0.5, 0));
        else if (scene == "dragon")  // TriangleMesh("model/dragon.txt", 1.5, Vec3(-5,-20,30), ..., 1) — main.cpp:292, glass material of :293
            extra[0].reset(new TriangleMesh(read_mesh_asset(assets + "/dragon.cgrtmesh", 1.5, Vec3(-5, -20, 30)), Vec3(1.0, 1.0, 1.0), 0.8, 0.5, 1));
        if (scene == "bunny" || scene == "dragon") objs.push_back(extra[0].get());

        cgrt_counters k;
        Image img = render(objs, opt, &k);  // main.cpp:401

        uint64_t h = 1469598103934665603ull;
        const unsigned char *b = reinterpret_cast<const unsigned char *>(img.rgb.data());
        for (size_t i = 0; i < img.rgb.size() * sizeof(double); i++) { h ^= b[i]; h *= 1099511628211ull; }
        double mean = 0;
        for (uint8_t v : img.rgb8) mean += v;
        mean /= (double)img.rgb8.size();
        std::FILE *fp = std::fopen(out.c_str(), "wb");  // the reference writes test.png through stb (main.cpp:412); PPM needs no codec
        if (!fp) { std::fprintf(stderr, "cannot write %s\n", out.c_str()); return 2; }
        std::fprintf(fp, "P6\n%d %d\n255\n", img.width, img.height);
        std::fwrite(img.rgb8.data(), 1, img.rgb8.size(), fp);
        std::fclose(fp);
        std::printf("%" PRIu64 " %" PRIu64 " %016" PRIx64 " %.6f\n", (uint64_t)k.hitpoints, (uint64_t)k.deposits, h, mean);
    } catch (const Error &e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return e.status == CGRT_ERR_NO_DEVICE ? 3 : 1;
    }
    return 0;
}
