// One timed vc::carveToMesh (ViewCache -> .off file: carve, average colour, handleUnseen, closure 3, marching cubes, writer) as
// a program, so that tools/mesh_bench.py --off can build it against two versions of include/voxcarve_host.hpp and alternate them.
// usage: carve_to_mesh_bench case.bin out.off   (case.bin: the layout tests/cpp/host_roundtrip.cpp reads); prints the time in ms
#include <chrono>
#include <cstdio>
#include <fstream>
#include <iostream>

#include "voxcarve_host.hpp"

int main(int argc, char** argv) {
    if (argc != 3) {
        std::cerr << "usage: " << argv[0] << " case.bin out.off" << std::endl;
        return 2;
    }
    std::ifstream in(argv[1], std::ios::binary);
    int32_t hdr[6];
    float s = 0.f;
    in.read((char*)hdr, sizeof hdr);
    in.read((char*)&s, sizeof s);
    vc::ViewCache c;
    c.V = hdr[3]; c.W = hdr[4]; c.H = hdr[5];
    c.P.resize((size_t)c.V * 12);
    c.M.resize((size_t)c.V * 12);
    c.mask_bits.resize((size_t)c.V * c.H * ((c.W + 31) / 32));
    c.images_bgr.resize((size_t)c.V * c.H * c.W * 3);
    in.read((char*)c.P.data(), c.P.size() * 4);
    in.read((char*)c.M.data(), c.M.size() * 4);
    in.read((char*)c.mask_bits.data(), c.mask_bits.size() * 4);
    in.read((char*)c.images_bgr.data(), c.images_bgr.size());
    if (!in) {
        std::cerr << "short case file" << std::endl;
        return 2;
    }
    const float t[3] = {0.5f, -0.25f, 2.0f};
    { vc::Engine warm(8, 8, 8, s); }  // CUDA context outside the timed call
    const auto t0 = std::chrono::steady_clock::now();
    const bool ok = vc::carveToMesh(c, hdr[0], hdr[1], hdr[2], s, VC_COLOR_AVG, 3, 1.5f, t, 0.5f, argv[2]);
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (!ok) return 1;
    std::printf("%.3f\n", ms);
    return 0;
}
