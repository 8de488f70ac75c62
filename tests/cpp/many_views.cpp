// A capture of more than 256 views through include/voxcarve_host.hpp: vc::carve into a stand-in of the reference Model, and
// vc::carveToMesh to an .off file.  tests/test_view_groups.py compares both with the oracle.
// usage: many_views case.bin model.bin mesh.off   (case.bin: the layout tests/cpp/host_roundtrip.cpp reads)
// model.bin: X*Y*Z bytes alpha != 0, then X*Y*Z bytes seen, in Model::flatten order.
#include <fstream>
#include <iostream>
#include <vector>

#include "voxcarve_host.hpp"

struct Vec4 {
    float v[4];
    Vec4() : v{0, 0, 0, 0} {}
    Vec4(float a, float b, float c, float d) : v{a, b, c, d} {}
    float operator()(int i) const { return v[i]; }
};

class MiniModel {  // the interface of the reference Model (Model.h:93-163) that the host layer uses
   public:
    MiniModel(int x, int y, int z, float size) : X(x), Y(y), Z(z), s(size), voxels((size_t)x * y * z, Vec4(50, 168, 141, 1)), seen((size_t)x * y * z, 0) {}
    int getX() { return X; }
    int getY() { return Y; }
    int getZ() { return Z; }
    float getSize() { return s; }
    Vec4 get(int x, int y, int z) { return voxels[flatten(x, y, z)]; }
    void set(int x, int y, int z, const Vec4& v) { voxels[flatten(x, y, z)] = v; }
    void see(int x, int y, int z) { seen[flatten(x, y, z)] = 1; }
    int X, Y, Z;
    float s;
    std::vector<Vec4> voxels;
    std::vector<char> seen;

   private:
    size_t flatten(int x, int y, int z) { return x + (size_t)X * (y + (size_t)Y * z); }
};

int main(int argc, char** argv) {
    if (argc != 4) {
        std::cerr << "usage: " << argv[0] << " case.bin model.bin mesh.off" << std::endl;
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
    try {
        MiniModel m(X, Y, Z, s);
        vc::carve(c, m);
        std::ofstream out(argv[2], std::ios::binary);
        for (const Vec4& v : m.voxels) out.put(v(3) != 0 ? 1 : 0);
        out.write(m.seen.data(), (std::streamsize)m.seen.size());
        const float t[3] = {0.5f, -0.25f, 2.0f};
        if (!vc::carveToMesh(c, X, Y, Z, s, VC_COLOR_AVG, 3, 1.5f, t, 0.5f, argv[3])) return 1;
    } catch (const std::exception& ex) {
        std::cerr << ex.what() << std::endl;
        return 1;
    }
    return 0;
}
