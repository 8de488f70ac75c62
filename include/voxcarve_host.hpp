// voxcarve_host.hpp — header-only C++17 host layer over the C ABI (voxcarve.h).
//
// Mirrors the reference's free functions for the hot path, templated on the model type so that it
// works with the reference's own `Model` (Model.h:93-163) unchanged and needs neither OpenCV nor
// Eigen to compile:
//     vc::carve / vc::fastCarve                          VoxelCarving.h:19,31
//     vc::reconstructClosestColor / reconstructAvgColor   ColorReconstruction.h:131,142
//     vc::marchingCubesClassify                           cube-index half of MarchingCubes.h:596
//     vc::applyClosure / vc::marchingCubes                Postprocessing3d.h:10, MarchingCubes.h:596 (incl. the .off writer)
// ModelT must offer what Model.h offers: getX(), getY(), getZ(), getSize(), get(x,y,z) returning a
// 4-vector with operator()(int) and a (float,float,float,float) constructor, set(x,y,z,vec), see(x,y,z).
// The per-dataset inputs the reference recomputes inside every call (estimatePoseFromImage +
// cv::undistort, VoxelCarving.cpp:25,36; ColorReconstruction.h:17-28) arrive cached in a ViewCache;
// voxcarve_shim.hpp builds one from (cameraMatrix, distCoeffs, images, masks) where OpenCV exists.
// Errors: the reference prints to std::cerr and returns; this layer throws vc::Error (message from
// vc_last_error) — nothing is ever computed on the CPU instead.
#ifndef VOXCARVE_HOST_HPP
#define VOXCARVE_HOST_HPP

#include <algorithm>
#include <cstdint>
#include <fstream>
#include <iostream>
#include <stdexcept>
#include <string>
#include <thread>
#include <type_traits>
#include <utility>
#include <vector>

#include "voxcarve.h"

namespace vc {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error("voxcarve error " + std::to_string(c) + ": " + m), code(c) {}
};

// Cached once per dataset (SURVEY §7-1).
struct ViewCache {
    int V = 0, W = 0, H = 0;
    std::vector<float> P;             // V*12: intr(CV_32F) * pose(3x4), first product of VoxelCarving.cpp:19
    std::vector<float> M;             // V*12: pose(3x4) world->camera (translation column = "camera", ColorReconstruction.h:21)
    std::vector<uint32_t> mask_bits;  // V*H*ceil(W/32), 1 = background; or ...
    std::vector<uint8_t> mask_bgr;    // ... V*H*W*3 undistorted 8UC3 masks (VoxelCarving.cpp:36)
    std::vector<uint8_t> images_bgr;  // V*H*W*3 undistorted images (ColorReconstruction.h:23); empty if no colouring
    // raw = true: mask_bgr / images_bgr are the DISTORTED 8UC3 inputs as cv::imread delivers them, and the engine runs
    // cv::undistort on the device (bit-exact with OpenCV's 8UC3 path) using K / dist from cameracalibration.yml
    bool raw = false;
    double K[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    std::vector<double> dist;         // k1 k2 p1 p2 [k3 [k4 k5 k6]]
};

// Result of a fresh carve in sparse form (vc_carve_download_sparse): a flag byte per 32x8x8-voxel brick of the slab, and the
// words of the listed bricks only.
struct SparseCarve {
    int X = 0, Y = 0, nz = 0;           // slab dimensions in voxels
    uint32_t nbx = 0, nby = 0, nbz = 0;  // bricks
    std::vector<uint8_t> flags;          // nbx*nby*nbz: 1 = carved whole, 2 = seen whole, 8 = listed
    std::vector<uint32_t> listed;        // brick index of every listed brick
    std::vector<uint32_t> words;         // 128 per listed brick: 64 occupied rows (8*plane + y), then 64 seen rows
};

struct McSummary {
    uint64_t hist[256];
    uint64_t active_cells, triangles;
};

class Engine {
   public:
    Engine(int X, int Y, int Z, float size, int z_begin = 0, int z_end = -1, int device = 0) : X_(X), Y_(Y), Z_(Z) {
        vc_grid_desc g{X, Y, Z, size, z_begin, z_end < 0 ? Z : z_end, device};
        int rc = vc_create(&g, &h_);
        if (rc != VC_OK) throw Error(rc, vc_last_error(nullptr));
        check(vc_slab_words(h_, &words_));
    }
    ~Engine() { vc_destroy(h_); }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;

    // all V views of the cache, up to VC_MAX_TOTAL_VIEWS: vc_set_views takes the first 256, vc_append_views the rest
    void setViews(const ViewCache& c, bool with_images) {
        if ((int)c.P.size() != c.V * 12) throw Error(VC_ERR_ARG, "ViewCache.P must hold V*12 floats");
        if (c.V > VC_MAX_TOTAL_VIEWS) throw Error(VC_ERR_ARG, "ViewCache holds " + std::to_string(c.V) + " views, more than VC_MAX_TOTAL_VIEWS");
        if (with_images && c.images_bgr.empty()) throw Error(VC_ERR_ARG, "colour reconstruction needs ViewCache.images_bgr");
        const int k = std::min(c.V, 256);
        check(vc_set_views(h_, k, c.W, c.H, c.P.data(), c.M.empty() ? nullptr : c.M.data()));
        if (c.raw) check(vc_set_calibration(h_, c.K, c.dist.data(), (int32_t)c.dist.size()));
        if (!c.mask_bits.empty()) check(vc_set_masks(h_, c.mask_bits.data(), VC_MASK_BITS));
        else if (!c.mask_bgr.empty()) check(vc_set_masks(h_, c.mask_bgr.data(), c.raw ? VC_MASK_BGR8_RAW : VC_MASK_BGR8));
        if (with_images) check(c.raw ? vc_set_images_raw(h_, c.images_bgr.data()) : vc_set_images(h_, c.images_bgr.data()));
        if (c.V > k) append(c, k, c.V, with_images);
        check(vc_synchronize(h_));  // the cache may be a temporary
    }
    // every view of `c` after the engine's current ones (same W x H; masks, M, raw-ness and images as the engine's own views)
    void appendViews(const ViewCache& c, bool with_images) {
        if ((int)c.P.size() != c.V * 12) throw Error(VC_ERR_ARG, "ViewCache.P must hold V*12 floats");
        append(c, 0, c.V, with_images);
    }
    void reset() { check(vc_reset(h_)); }
    void carve(int mode = VC_EXACT, int v0 = 0, int v1 = -1) { check(vc_carve(h_, mode, v0, v1, 0)); }
    // carve all views + download both volumes, the D2H of finished z-chunks overlapped with the carving of the next
    void carveDownload(std::vector<uint32_t>& occ, std::vector<uint32_t>& seen, int mode = VC_EXACT) {
        occ.resize(words_);
        seen.resize(words_);
        check(vc_carve_download(h_, mode, occ.data(), seen.data(), words_));
    }
    // fresh carve + sparse download (vc_reset is implied): 1/25 of the PCIe bytes of carveDownload on a 1024^3 grid
    void carveDownloadSparse(SparseCarve& sp) {
        check(vc_reset(h_));
        check(vc_sparse_dims(h_, &sp.nbx, &sp.nby, &sp.nbz));
        sp.X = X_; sp.Y = Y_; sp.nz = (int)(words_ / ((uint64_t)Y_ * wordsPerRow()));
        const uint64_t nb = (uint64_t)sp.nbx * sp.nby * sp.nbz;
        sp.flags.resize(nb);
        uint64_t cap = std::max<uint64_t>(1024, nb / 16), n = 0;
        for (int attempt = 0;; attempt++) {
            sp.listed.resize(cap);
            sp.words.resize(cap * 128);
            const int rc = vc_carve_download_sparse(h_, sp.flags.data(), nb, sp.listed.data(), sp.words.data(), cap, &n);
            if (rc == VC_ERR_CAPACITY && n > cap && attempt == 0) {  // more listed bricks than guessed: the volumes are complete on the device,
                cap = n;                                              // ask again with room (a reset + second carve: rare, and still exact)
                check(vc_reset(h_));
                continue;
            }
            check(rc);
            break;
        }
        sp.listed.resize(n);
        sp.words.resize(n * 128);
    }
    void fastCarve(int mode = VC_EXACT) { check(vc_fast_carve(h_, mode)); }
    void color(int mode) { check(vc_color(h_, mode)); }
    // occlusion-aware colouring (vc_color_visible): a surface voxel takes its colour only from the views that see it
    void colorVisible(int mode, float tolerance = 2.0f) { check(vc_color_visible(h_, mode, tolerance)); }
    McSummary mcClassify() {
        McSummary s{};
        check(vc_mc_classify(h_));
        check(vc_download_mc(h_, s.hist, &s.active_cells, &s.triangles));
        return s;
    }
    std::vector<uint32_t> occupied() { std::vector<uint32_t> w(words_); check(vc_download_occupied(h_, w.data(), words_)); return w; }
    std::vector<uint32_t> seen() { std::vector<uint32_t> w(words_); check(vc_download_seen(h_, w.data(), words_)); return w; }
    void upload(const std::vector<uint32_t>& occ, const std::vector<uint32_t>& seen) { check(vc_upload_volumes(h_, occ.data(), seen.data(), words_)); }
    void colors(std::vector<uint64_t>& idx, std::vector<uint8_t>& rgbn) {
        uint64_t n = 0;
        check(vc_surface_count(h_, &n));
        idx.resize(n);
        rgbn.resize(n * 4);
        check(vc_download_colors(h_, idx.data(), rgbn.data(), n));
    }
    // "next" rows: dense RGBA Model on the device
    void denseUpload(const std::vector<float>& rgba) { check(vc_dense_upload(h_, rgba.data())); }
    void denseApplyCarved() { check(vc_dense_apply_carved(h_)); }
    void denseClosure(int kernelSize) { check(vc_dense_closure(h_, kernelSize)); }
    void denseDownload(std::vector<float>& rgba) { check(vc_dense_download(h_, rgba.data())); }
    // mesh left on the device (for formatOff); returns the triangle count
    uint64_t mcMesh(float threshold) { uint64_t n = 0; check(vc_mc_mesh(h_, threshold, &n)); return n; }
    uint64_t mcMesh(float threshold, std::vector<float>& verts, std::vector<uint32_t>& rgb) {
        const uint64_t n = mcMesh(threshold);
        verts.resize(n * 9);
        rgb.resize(n * 3);
        check(vc_download_mesh(h_, verts.data(), rgb.data(), n));
        return n;
    }
    // marchingCubes of the Model denseFromVolumes(applyColors, handleUnseen) [+ denseClosure(closureK)] would build, from the bit
    // volumes and colour records without the dense Model (closureK = 0: no closure); same triangles as that chain + mcMesh
    uint64_t meshFromVolumes(bool applyColors, bool handleUnseen, int closureK, float threshold) {
        uint64_t n = 0;
        check(vc_mesh_from_volumes(h_, applyColors ? 1 : 0, handleUnseen ? 1 : 0, closureK, threshold, &n));
        return n;
    }
    uint64_t meshFromVolumes(bool applyColors, bool handleUnseen, int closureK, float threshold, std::vector<float>& verts,
                             std::vector<uint32_t>& rgb) {
        const uint64_t n = meshFromVolumes(applyColors, handleUnseen, closureK, threshold);
        verts.resize(n * 9);
        rgb.resize(n * 3);
        check(vc_download_mesh(h_, verts.data(), rgb.data(), n));
        return n;
    }
    // the .off text of the mesh on the device (vertex = index coordinates * scale + t), formatted there; returns its size in
    // bytes.  downloadOff copies bytes [offset, offset + n) of it.
    uint64_t formatOff(float scale, float tx, float ty, float tz) { uint64_t n = 0; check(vc_mesh_format_off(h_, scale, tx, ty, tz, &n)); return n; }
    void downloadOff(uint64_t offset, void* dst, uint64_t n) { check(vc_download_mesh_off(h_, offset, dst, n)); }
    // multi-GPU plumbing: balanced z-slabs, one-plane halos, NCCL collectives inside the library (voxcarve.h)
    std::vector<int32_t> planSlabs(int n_parts) { std::vector<int32_t> b((size_t)n_parts + 1); check(vc_plan_slabs(h_, n_parts, b.data())); return b; }
    void setSlab(int z_begin, int z_end) { check(vc_set_slab(h_, z_begin, z_end)); check(vc_slab_words(h_, &words_)); }
    void allocFullVolumes() { check(vc_alloc_full_volumes(h_)); }
    void commInit(int rank, int world, const void* unique_id_128) { check(vc_comm_init(h_, rank, world, unique_id_128)); }
    void exchangeHalos() { check(vc_exchange_halos(h_)); }
    void gather(const std::vector<int32_t>& z_bounds, int what = 1) { check(vc_gather(h_, what, z_bounds.data())); }
    // engines of this process: everyone pulls the other slabs over NVLink (no NCCL); e.g. before fastCarve-style whole-grid work
    static void gatherPeer(const std::vector<Engine*>& engines, int what = 1) {
        std::vector<vc_engine*> hs;
        for (Engine* e : engines) hs.push_back(e->handle());
        if (hs.empty()) return;
        const int rc = vc_gather_peer(hs.data(), (int32_t)hs.size(), what);
        if (rc != VC_OK) throw Error(rc, vc_last_error(hs[0]));
    }
    void allreduce(uint64_t* values, int n) { check(vc_comm_allreduce_u64(h_, values, n)); }
    std::vector<uint32_t> downloadFull(int which) {
        std::vector<uint32_t> w((size_t)Z_ * Y_ * wordsPerRow());
        check(vc_download_full(h_, which, w.data(), w.size()));
        return w;
    }
    void synchronize() { check(vc_synchronize(h_)); }
    // download this slab's volumes into caller memory (e.g. at the slab's offset inside whole-grid host vectors)
    void carveDownloadInto(uint32_t* occ, uint32_t* seen, int mode = VC_EXACT) { check(vc_carve_download(h_, mode, occ, seen, words_)); }
    uint64_t slabWords() const { return words_; }
    vc_stats stats() { vc_stats s{}; check(vc_get_stats(h_, &s)); return s; }
    vc_engine* handle() { return h_; }
    int wordsPerRow() const { return (X_ + 31) / 32; }

   private:
    void check(int rc) { if (rc != VC_OK) throw Error(rc, vc_last_error(h_)); }
    void append(const ViewCache& c, int v0, int v1, bool with_images) {
        const size_t bgr = (size_t)c.H * c.W * 3, words = (size_t)c.H * ((c.W + 31) / 32);
        if (with_images && c.images_bgr.empty()) throw Error(VC_ERR_ARG, "colour reconstruction needs ViewCache.images_bgr");
        const void* masks = !c.mask_bits.empty() ? (const void*)(c.mask_bits.data() + v0 * words) : (const void*)(c.mask_bgr.data() + v0 * bgr);
        const int fmt = !c.mask_bits.empty() ? VC_MASK_BITS : (c.raw ? VC_MASK_BGR8_RAW : VC_MASK_BGR8);
        check(vc_append_views(h_, v1 - v0, c.P.data() + (size_t)v0 * 12, c.M.empty() ? nullptr : c.M.data() + (size_t)v0 * 12, masks, fmt,
                              with_images ? c.images_bgr.data() + v0 * bgr : nullptr));
    }
    vc_engine* h_ = nullptr;
    uint64_t words_ = 0;
    int X_, Y_, Z_;
};

namespace detail {
template <class ModelT>
using Vec4Of = std::decay_t<decltype(std::declval<ModelT&>().get(0, 0, 0))>;

// device bit volumes -> the reference Model: set(x,y,z,(0,0,0,0)) for carved voxels (VoxelCarving.cpp:52), see() (:54)
template <class ModelT>
void applyCarve(ModelT& model, const std::vector<uint32_t>& occ, const std::vector<uint32_t>& seen) {
    const int X = model.getX(), Y = model.getY(), Z = model.getZ(), Wx = (X + 31) / 32;
    const Vec4Of<ModelT> zero(0.f, 0.f, 0.f, 0.f);
    for (int z = 0; z < Z; z++)
        for (int y = 0; y < Y; y++)
            for (int x = 0; x < X; x++) {
                const size_t w = ((size_t)z * Y + y) * Wx + (x >> 5);
                if (!((occ[w] >> (x & 31)) & 1u)) model.set(x, y, z, zero);
                if ((seen[w] >> (x & 31)) & 1u) model.see(x, y, z);
            }
}

// sparse result of a fresh carve -> the reference Model, brick by brick: a carved brick clears and sees all its voxels, a seen
// brick sees them, an untouched one costs nothing, a listed one is applied bit by bit
template <class ModelT>
void applyCarveSparse(ModelT& model, const SparseCarve& sp, int z_begin = 0) {
    const Vec4Of<ModelT> zero(0.f, 0.f, 0.f, 0.f);
    std::vector<int64_t> slot((size_t)sp.nbx * sp.nby * sp.nbz, -1);
    for (size_t i = 0; i < sp.listed.size(); i++) slot[sp.listed[i]] = (int64_t)i;
    for (uint32_t bz = 0; bz < sp.nbz; bz++)
        for (uint32_t by = 0; by < sp.nby; by++)
            for (uint32_t bx = 0; bx < sp.nbx; bx++) {
                const size_t b = ((size_t)bz * sp.nby + by) * sp.nbx + bx;
                const uint8_t f = sp.flags[b];
                if (!(f & (1 | 2 | 8))) continue;
                const int x0 = (int)bx * 32, x1 = std::min(x0 + 32, sp.X), y0 = (int)by * 8, y1 = std::min(y0 + 8, sp.Y), z0 = (int)bz * 8, z1 = std::min(z0 + 8, sp.nz);
                const uint32_t* w = (f & 8) ? &sp.words[(size_t)slot[b] * 128] : nullptr;
                for (int z = z0; z < z1; z++)
                    for (int y = y0; y < y1; y++) {
                        const uint32_t o = w ? w[(z - z0) * 8 + (y - y0)] : ((f & 1) ? 0u : 0xffffffffu);
                        const uint32_t sn = w ? w[64 + (z - z0) * 8 + (y - y0)] : ((f & 2) ? 0xffffffffu : 0u);
                        for (int x = x0; x < x1; x++) {
                            if (!((o >> (x & 31)) & 1u)) model.set(x, y, z_begin + z, zero);
                            if ((sn >> (x & 31)) & 1u) model.see(x, y, z_begin + z);
                        }
                    }
            }
}

// sparse result -> the plain bit volumes (what carveDownload delivers)
inline void expandSparse(const SparseCarve& sp, std::vector<uint32_t>& occ, std::vector<uint32_t>& seen) {
    const int Wx = (sp.X + 31) / 32;
    occ.assign((size_t)sp.nz * sp.Y * Wx, 0u);
    seen.assign(occ.size(), 0u);
    std::vector<int64_t> slot((size_t)sp.nbx * sp.nby * sp.nbz, -1);
    for (size_t i = 0; i < sp.listed.size(); i++) slot[sp.listed[i]] = (int64_t)i;
    for (uint32_t bz = 0; bz < sp.nbz; bz++)
        for (uint32_t by = 0; by < sp.nby; by++)
            for (uint32_t bx = 0; bx < sp.nbx; bx++) {
                const size_t b = ((size_t)bz * sp.nby + by) * sp.nbx + bx;
                const uint8_t f = sp.flags[b];
                const int rem = sp.X - (int)bx * 32;
                const uint32_t valid = rem >= 32 ? 0xffffffffu : ((1u << rem) - 1u);
                const uint32_t* w = (f & 8) ? &sp.words[(size_t)slot[b] * 128] : nullptr;
                for (int z = (int)bz * 8; z < std::min((int)bz * 8 + 8, sp.nz); z++)
                    for (int y = (int)by * 8; y < std::min((int)by * 8 + 8, sp.Y); y++) {
                        const size_t i = ((size_t)z * sp.Y + y) * Wx + bx;
                        const int r = (z - (int)bz * 8) * 8 + (y - (int)by * 8);
                        occ[i] = w ? w[r] : ((f & 1) ? 0u : valid);
                        seen[i] = w ? w[64 + r] : ((f & 2) ? valid : 0u);
                    }
            }
}

// occupancy of an existing Model (alpha != 0) -> bit volume, for the colour / MC passes
template <class ModelT>
std::vector<uint32_t> packOccupancy(ModelT& model) {
    const int X = model.getX(), Y = model.getY(), Z = model.getZ(), Wx = (X + 31) / 32;
    std::vector<uint32_t> occ((size_t)Z * Y * Wx, 0u);
    for (int z = 0; z < Z; z++)
        for (int y = 0; y < Y; y++)
            for (int x = 0; x < X; x++)
                if (model.get(x, y, z)(3) != 0) occ[((size_t)z * Y + y) * Wx + (x >> 5)] |= 1u << (x & 31);
    return occ;
}

// the Model's voxels as X*Y*Z*4 floats in Model::flatten order (Model.h:104-106)
template <class ModelT>
std::vector<float> packVoxels(ModelT& model) {
    const int X = model.getX(), Y = model.getY(), Z = model.getZ();
    std::vector<float> rgba((size_t)X * Y * Z * 4);
    for (int z = 0; z < Z; z++)
        for (int y = 0; y < Y; y++)
            for (int x = 0; x < X; x++) {
                const auto v = model.get(x, y, z);
                float* o = &rgba[4 * ((size_t)x + (size_t)X * ((size_t)y + (size_t)Y * z))];
                o[0] = v(0); o[1] = v(1); o[2] = v(2); o[3] = v(3);
            }
    return rgba;
}

template <class ModelT>
void colorPass(const ViewCache& views, ModelT& model, int mode) {
    Engine e(model.getX(), model.getY(), model.getZ(), model.getSize());
    e.setViews(views, true);
    const std::vector<uint32_t> occ = packOccupancy(model);
    e.upload(occ, std::vector<uint32_t>(occ.size(), 0u));
    e.color(mode);
    std::vector<uint64_t> idx;
    std::vector<uint8_t> rgbn;
    e.colors(idx, rgbn);
    const uint64_t X = model.getX(), Y = model.getY();
    for (size_t i = 0; i < idx.size(); i++) {
        if (rgbn[i * 4 + 3] == 0) continue;  // no observation: voxel untouched (ColorReconstruction.cpp:29-31)
        const int x = (int)(idx[i] % X), y = (int)((idx[i] / X) % Y), z = (int)(idx[i] / (X * Y));
        model.set(x, y, z, Vec4Of<ModelT>((float)rgbn[i * 4], (float)rgbn[i * 4 + 1], (float)rgbn[i * 4 + 2], 1.f));
    }
}

// SimpleMesh::WriteMesh (MarchingCubes.h:59-87) for a triangle soup in host memory: vertex = index coordinates
// * (scale * voxel size) + translation (MarchingCubes.h:561-566), default ostream float formatting.  Kept for triangles already in
// host memory and as the host writer the device text is tested against; the functions below use the overload that follows.
inline bool writeOff(const std::string& outFileName, uint64_t nt, const std::vector<float>& verts, const std::vector<uint32_t>& rgb,
                     float sf, float tx, float ty, float tz) {
    std::ofstream outFile(outFileName);
    if (!outFile.is_open()) return false;
    outFile << "OFF" << std::endl;
    outFile << nt * 3 << " " << nt << " 0" << std::endl;
    for (uint64_t i = 0; i < nt * 3; i++)
        outFile << verts[i * 3] * sf + tx << " " << verts[i * 3 + 1] * sf + ty << " " << verts[i * 3 + 2] * sf + tz << std::endl;
    for (uint64_t i = 0; i < nt; i++)
        outFile << "3 " << 3 * i << " " << 3 * i + 1 << " " << 3 * i + 2 << " " << rgb[i * 3] << " " << rgb[i * 3 + 1] << " " << rgb[i * 3 + 2] << std::endl;
    outFile.close();
    return true;
}

// SimpleMesh::WriteMesh for the mesh on the device: the text is formatted there (vc_mesh_format_off), downloaded in chunks of
// 64 MiB through one buffer and written with ofstream::write.  false if the file cannot be opened or written.
inline bool writeOff(Engine& e, const std::string& outFileName, float sf, float tx, float ty, float tz) {
    const uint64_t n = e.formatOff(sf, tx, ty, tz);
    std::ofstream outFile(outFileName, std::ios::binary);
    if (!outFile.is_open()) return false;
    std::vector<char> buf((size_t)std::min<uint64_t>(n, 64ull << 20));
    for (uint64_t o = 0; o < n && outFile; o += buf.size()) {
        const uint64_t k = std::min<uint64_t>(buf.size(), n - o);
        e.downloadOff(o, buf.data(), k);
        outFile.write(buf.data(), (std::streamsize)k);
    }
    outFile.close();
    return !outFile.fail();
}
}  // namespace detail

// carve() — VoxelCarving.cpp:60-72.  With intermediateMeshes the Model's mesh after every view goes to
// <intermediateDir>/image_<i>_mesh.off, translated by i * (X + 2) * size along x, exactly as :65-68 writes it (the directory
// must exist: main.cpp:47 creates ./out/intermediate); `perView` (if given) also receives the cube-index summary per view.
template <class ModelT>
void carve(const ViewCache& views, ModelT& model, bool intermediateMeshes = false, std::vector<McSummary>* perView = nullptr,
           const std::string& intermediateDir = "out/intermediate") {
    std::cout << "LOG - VC: starting carving process (version 1)." << std::endl;
    Engine e(model.getX(), model.getY(), model.getZ(), model.getSize());
    e.setViews(views, false);
    std::vector<uint32_t> occ, seen;
    if (intermediateMeshes) {
        e.denseUpload(detail::packVoxels(model));  // the Model as it is now (colours, earlier carves)
        for (int i = 0; i < views.V; i++) {
            e.carve(VC_EXACT, i, i + 1);
            std::cout << "LOG - VC: generating intermediate mesh for image " << i << std::endl;
            e.denseApplyCarved();
            e.mcMesh(0.5f);
            const float tx = (float)(i * (model.getX() + 2)) * model.getSize();  // Vector3f(i*(model.getX() + 2)*model.getSize(), 0, 0)
            if (!detail::writeOff(e, intermediateDir + "/image_" + std::to_string(i) + "_mesh.off", 1.0f * model.getSize(), tx, 0.f, 0.f))
                std::cout << "ERR - MC: unable to write output file!" << std::endl;  // the reference carries on (its bool result is ignored)
            if (perView) perView->push_back(e.mcClassify());
        }
        occ = e.occupied();
        seen = e.seen();
        detail::applyCarve(model, occ, seen);
    } else {  // the common case: sparse download (a few % of the bytes), applied brick by brick
        SparseCarve sp;
        e.carveDownloadSparse(sp);
        detail::applyCarveSparse(model, sp);
    }
    std::cout << "LOG - VC: carving complete." << std::endl;
}

// carve() on several GPUs of this host: the grid is cut into balanced z-slabs (vc_plan_slabs), one engine and one host
// thread per device, every engine sees all views; each slab comes back from its GPU in sparse form (one PCIe link per GPU, no
// device-to-device traffic: a host Model needs no all-gather) and is applied to the Model.  Same Model as carve().
template <class ModelT>
void carveOnDevices(const ViewCache& views, ModelT& model, const std::vector<int>& devices) {
    if (devices.size() <= 1) {
        carve(views, model);
        return;
    }
    std::cout << "LOG - VC: starting carving process (version 1)." << std::endl;
    const int X = model.getX(), Y = model.getY(), Z = model.getZ(), n = (int)std::min<size_t>(devices.size(), (size_t)Z);
    const float size = model.getSize();
    std::vector<SparseCarve> parts((size_t)n);
    std::vector<int32_t> bounds;
    {
        Engine planner(X, Y, Z, size, 0, -1, devices[0]);
        planner.setViews(views, false);
        bounds = planner.planSlabs(n);
    }
    std::vector<std::string> errors((size_t)n);
    std::vector<std::thread> threads;
    for (int r = 0; r < n; r++)
        threads.emplace_back([&, r] {
            try {
                Engine e(X, Y, Z, size, bounds[r], bounds[r + 1], devices[r]);
                e.setViews(views, false);
                e.carveDownloadSparse(parts[r]);
            } catch (const std::exception& ex) {
                errors[r] = ex.what();
            }
        });
    for (auto& t : threads) t.join();
    for (const auto& m : errors)
        if (!m.empty()) throw Error(VC_ERR_CUDA, m);
    for (int r = 0; r < n; r++) detail::applyCarveSparse(model, parts[r], bounds[r]);  // one thread: Model::seen is a vector<bool>
    std::cout << "LOG - VC: carving complete." << std::endl;
}

// fastCarve() — VoxelCarving.cpp:74-167
template <class ModelT>
void fastCarve(const ViewCache& views, ModelT& model) {
    std::cout << "LOG - VC: starting carving process (version 2)." << std::endl;
    Engine e(model.getX(), model.getY(), model.getZ(), model.getSize());
    e.setViews(views, false);
    e.fastCarve();
    detail::applyCarve(model, e.occupied(), e.seen());
    std::cout << "LOG - VC: carving complete." << std::endl;
}

// reconstructClosestColor() — ColorReconstruction.cpp:22-46
template <class ModelT>
void reconstructClosestColor(const ViewCache& views, ModelT& model) {
    std::cout << "LOG - CR: starting color reconstruction (closest color)." << std::endl;
    detail::colorPass(views, model, VC_COLOR_CLOSEST);
    std::cout << "LOG - CR: color reconstruction finished." << std::endl;
}

// reconstructAvgColor() — ColorReconstruction.cpp:48-70
template <class ModelT>
void reconstructAvgColor(const ViewCache& views, ModelT& model) {
    std::cout << "LOG - CR: starting color reconstruction (average color)." << std::endl;
    detail::colorPass(views, model, VC_COLOR_AVG);
    std::cout << "LOG - CR: color reconstruction finished." << std::endl;
}

// cube-index classification of marchingCubes() — MarchingCubes.cpp:12-18, MarchingCubes.h:479-488
template <class ModelT>
McSummary marchingCubesClassify(ModelT& model) {
    std::cout << "LOG - MC: starting to process Voxels." << std::endl;
    Engine e(model.getX(), model.getY(), model.getZ(), model.getSize());
    const std::vector<uint32_t> occ = detail::packOccupancy(model);
    e.upload(occ, std::vector<uint32_t>(occ.size(), 0u));
    const McSummary s = e.mcClassify();
    std::cout << "LOG - MC: voxel processing completed." << std::endl;
    return s;
}

// applyClosure() — Postprocessing3d.h:10, Postprocessing3d.cpp:4-100. Returns -1 for an even kernel size, like the reference.
template <class ModelT>
int applyClosure(ModelT* model, int kernelSize) {
    std::cout << "LOG - PP: starting postprocessing." << std::endl;
    if (kernelSize % 2 != 1) {
        std::cerr << "Invalid kernel size for post processing, skipping..." << std::endl;
        return -1;
    }
    const int X = model->getX(), Y = model->getY(), Z = model->getZ();
    Engine e(X, Y, Z, model->getSize());
    std::vector<float> rgba = detail::packVoxels(*model);
    e.denseUpload(rgba);
    e.denseClosure(kernelSize);
    e.denseDownload(rgba);
    for (int z = 0; z < Z; z++)
        for (int y = 0; y < Y; y++)
            for (int x = 0; x < X; x++) {
                const float* o = &rgba[4 * ((size_t)x + (size_t)X * ((size_t)y + (size_t)Y * z))];
                model->set(x, y, z, detail::Vec4Of<ModelT>(o[0], o[1], o[2], o[3]));
            }
    std::cout << "LOG - PP: postprocessing completed." << std::endl;
    return 0;
}

// marchingCubes() — MarchingCubes.h:596, MarchingCubes.cpp:8-31 + SimpleMesh::WriteMesh MarchingCubes.h:59-87.
// translation = {tx, ty, tz}. Returns false if the file cannot be written.
template <class ModelT>
bool marchingCubes(ModelT* model, float scale = 1.0f, const float* translation = nullptr, float threshold = 0.5f,
                   const std::string& outFileName = "out/mesh.off") {
    std::cout << "LOG - MC: starting to process Voxels." << std::endl;
    Engine e(model->getX(), model->getY(), model->getZ(), model->getSize());
    e.denseUpload(detail::packVoxels(*model));
    e.mcMesh(threshold);
    std::cout << "LOG - MC: voxel processing completed.\n Writing mesh..." << std::endl;
    const float sf = scale * model->getSize();
    const float tx = translation ? translation[0] : 0.f, ty = translation ? translation[1] : 0.f, tz = translation ? translation[2] : 0.f;
    if (!detail::writeOff(e, outFileName, sf, tx, ty, tz)) {
        std::cout << "ERR - MC: unable to write output file!" << std::endl;
        return false;
    }
    std::cout << "LOG - MC: Mesh written, marchingCubes completed." << std::endl;
    return true;
}

// main.cpp:260-303 from a ViewCache to the .off file, without a host Model: carve -> [reconstructClosestColor (colorMode 1) /
// reconstructAvgColor (2)] -> handleUnseen -> [applyClosure(closureK), closureK = 0: none] -> marchingCubes(scale, translation,
// threshold).  The volumes, colour records and mesh stay on the device, and the .off text is formatted there too, so grids whose
// dense Model does not fit the GPU (2048^3: 128 GiB) are meshed too, and only the file's bytes cross PCIe.  Returns false if the file cannot be written.
// visibilityTolerance = nullptr colours as the reference does (every view whose image holds the voxel's pixel); a tolerance in
// voxel sizes colours each surface voxel from the views that see it (vc_color_visible).
inline bool carveToMesh(const ViewCache& views, int X, int Y, int Z, float size, int colorMode, int closureK, float scale = 1.0f,
                        const float* translation = nullptr, float threshold = 0.5f, const std::string& outFileName = "out/mesh.off",
                        int device = 0, const float* visibilityTolerance = nullptr) {
    Engine e(X, Y, Z, size, 0, -1, device);
    e.setViews(views, colorMode != 0);
    e.carve();
    if (colorMode && visibilityTolerance) e.colorVisible(colorMode, *visibilityTolerance);
    else if (colorMode) e.color(colorMode);
    e.meshFromVolumes(colorMode != 0, true, closureK, threshold);
    const float tx = translation ? translation[0] : 0.f, ty = translation ? translation[1] : 0.f, tz = translation ? translation[2] : 0.f;
    if (!detail::writeOff(e, outFileName, scale * size, tx, ty, tz)) {
        std::cout << "ERR - MC: unable to write output file!" << std::endl;
        return false;
    }
    return true;
}

}  // namespace vc
#endif  // VOXCARVE_HOST_HPP
