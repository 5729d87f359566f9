// rays1_main.cpp -- the reference's executable surface: `./rays1_b200 [-w] [-n N]` renders small, medium and large,
// prints the reference's report blocks and writes out_<scene>.txt (and out_<scene>.tga with -w), exactly as
// src/latest/rayweek1.cpp:930-988 does.  Extra flags (not in the reference) select what it fixes at compile time:
//   --gpus N  --variant mega|wavefront|packed|tensor|tensor-stream|bvh|scalar|coop|deferred|dual  --width W --height H --spp S --bounces B  --scene NAME (repeatable)
//   --scene-file PATH (text scene description, see rays1_host.cpp)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "rays1_host.h"

int main(int argc, const char *argv[])
{
    bool write_tga = false;
    int num_runs = 1;
    const static int MAX_NUMS = 32;
    RESULT results[MAX_NUMS];
    std::vector<std::string> scenes;
    HostConfig &cfg = host_config();

    for (int i = 1; i < argc; ++i) {
        auto next_int = [&](int lo) { int v = (i + 1 < argc) ? atoi(argv[++i]) : 0; if (v < lo) { printf("Invalid value for %s\n", argv[i - 1]); exit(2); } return v; };
        if (strcmp(argv[i], "-w") == 0) write_tga = true;
        else if (strcmp(argv[i], "-n") == 0 && i + 1 < argc) {  // rayweek1.cpp:948-957
            int n = atoi(argv[++i]);
            if (n >= 1 && n < MAX_NUMS) num_runs = n;
            else printf("Invalid num_runs parameter: %d\n", n);
        } else if (strcmp(argv[i], "--gpus") == 0) cfg.n_gpus = next_int(1);
        else if (strcmp(argv[i], "--width") == 0) cfg.width = next_int(1);
        else if (strcmp(argv[i], "--height") == 0) cfg.height = next_int(1);
        else if (strcmp(argv[i], "--spp") == 0) cfg.spp = next_int(1);
        else if (strcmp(argv[i], "--bounces") == 0) cfg.max_bounces = next_int(0);
        else if (strcmp(argv[i], "--seed") == 0) cfg.seed = (uint32_t)next_int(0);
        else if (strcmp(argv[i], "--scene") == 0 && i + 1 < argc) scenes.push_back(argv[++i]);
        else if (strcmp(argv[i], "--scene-file") == 0 && i + 1 < argc) scenes.push_back(std::string("@") + argv[++i]);
        else if (strcmp(argv[i], "--variant") == 0 && i + 1 < argc) {
            const char *v = argv[++i];
            if (!strcmp(v, "mega")) cfg.variant = R1_VARIANT_MEGAKERNEL;
            else if (!strcmp(v, "wavefront")) cfg.variant = R1_VARIANT_WAVEFRONT;
            else if (!strcmp(v, "scalar")) cfg.variant = R1_VARIANT_MEGAKERNEL_SCALAR;
            else if (!strcmp(v, "coop")) cfg.variant = R1_VARIANT_MEGAKERNEL_COOP;
            else if (!strcmp(v, "deferred")) cfg.variant = R1_VARIANT_MEGAKERNEL_DEFERRED;
            else if (!strcmp(v, "dual")) cfg.variant = R1_VARIANT_MEGAKERNEL_DUAL;
            else if (!strcmp(v, "tensor")) cfg.variant = R1_VARIANT_MEGAKERNEL_TENSOR;
            else if (!strcmp(v, "tensor-stream")) cfg.variant = R1_VARIANT_MEGAKERNEL_TENSOR_STREAM;
            else if (!strcmp(v, "packed")) cfg.variant = R1_VARIANT_MEGAKERNEL_PACKED;
            else if (!strcmp(v, "bvh")) cfg.variant = R1_VARIANT_MEGAKERNEL_BVH;
            else { printf("Invalid variant: %s\n", v); exit(2); }
        }
    }
    if (scenes.empty()) scenes = { "small", "medium", "large" };  // rayweek1.cpp:969-984

    Pix *pixels = new Pix[(size_t)cfg.width * cfg.height];
    memset(pixels, 0, sizeof(Pix) * (size_t)cfg.width * cfg.height);

    const char *version = "b200";
    for (const std::string &name : scenes) {
        for (int i = 0; i < num_runs; ++i) {
            // "@path" = a scene description file; it is reported under the file's base name
            Scene *scene = name[0] == '@' ? create_scene_from_file(name.c_str() + 1) : create_scene_by_name(name.c_str());
            if (!scene) { printf("Unknown scene: %s\n", name.c_str()); return 2; }
            std::string label = name;
            if (name[0] == '@') {
                label = name.substr(name.find_last_of('/') == std::string::npos ? 1 : name.find_last_of('/') + 1);
                label = label.substr(0, label.find('.'));
            }
            results[i] = benchmark(scene, pixels, write_tga, label.c_str());
            if (i == num_runs - 1) log_results(version, label.c_str(), results, num_runs);
        }
    }
    delete[] pixels;
    return 0;
}
