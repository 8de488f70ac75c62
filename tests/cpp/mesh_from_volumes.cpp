// vc::carveToMesh (main.cpp:260-303 without a host Model) next to the same chain through the dense Model on the device
// (vc_dense_from_volumes -> vc_dense_closure -> vc_mc_mesh); both write .off files that tests/test_mesh_from_volumes.py compares.
// usage: mesh_from_volumes case.bin sparse.off dense.off   (case.bin: the layout tests/cpp/host_roundtrip.cpp reads)
#include <cstdio>
#include <fstream>
#include <iostream>

#include "voxcarve_host.hpp"

int main(int argc, char** argv) {
    if (argc != 4) {
        std::cerr << "usage: " << argv[0] << " case.bin sparse.off dense.off" << std::endl;
        return 2;
    }
    std::ifstream in(argv[1], std::ios::binary);
    int32_t hdr[6];
    float s = 0.f;
    in.read((char*)hdr, sizeof hdr);
    in.read((char*)&s, sizeof s);
    const int X = hdr[0], Y = hdr[1], Z = hdr[2];
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
    try {
        if (!vc::carveToMesh(c, X, Y, Z, s, VC_COLOR_AVG, 3, 1.5f, t, 0.5f, argv[2])) return 1;
        vc::Engine e(X, Y, Z, s);
        e.setViews(c, true);
        e.carve();
        e.color(VC_COLOR_AVG);
        if (vc_dense_from_volumes(e.handle(), 1, 1) != VC_OK) throw vc::Error(VC_ERR_STATE, vc_last_error(e.handle()));
        e.denseClosure(3);
        std::vector<float> verts;
        std::vector<uint32_t> rgb;
        const uint64_t nt = e.mcMesh(0.5f, verts, rgb);
        if (!vc::detail::writeOff(argv[3], nt, verts, rgb, 1.5f * s, t[0], t[1], t[2])) return 1;
    } catch (const std::exception& ex) {
        std::cerr << ex.what() << std::endl;
        return 1;
    }
    return 0;
}
