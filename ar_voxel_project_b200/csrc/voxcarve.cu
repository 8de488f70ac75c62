// voxcarve.cu — engine and C ABI (include/voxcarve.h) of the B200-native voxel-carving path.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
// There is no CPU path in this library: every entry point needs a CUDA device.
#include "../../include/voxcarve.h"

#include <cuda.h>             // types only: the few driver entry points used (vol_alloc) are fetched with cudaGetDriverEntryPoint
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>             // types and prototypes only: the library is dlopen-ed by vc_comm_init (see load_nccl)
#include <nvtx3/nvToolsExt.h>  // header-only; ranges named after the reference's Benchmark phases (Benchmark.h:86-124)

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "mc_tables.inc"
#include "vc_kernels.cuh"

static_assert(VC_MESH_MAX_CLOSURE == 2 * VC_CLOSURE_SMAX + 1, "vc_dilate_kernel's plane window holds 2 * VC_CLOSURE_SMAX + 1 planes");

namespace {

std::string g_create_error;
std::mutex g_const_mutex;
// which (engine uid, views version, view group) currently owns c_view / c_cam on each device
// and an event recorded after the owner's last launch that reads them: a new owner waits for it before overwriting the symbols
struct ConstOwner { unsigned long long uid = 0, version = 0; int group = 0; cudaEvent_t last_use = nullptr; bool used = false; };
ConstOwner g_const_owner[64];
unsigned long long g_next_uid = 1;

}  // namespace

extern "C" {
static cudaError_t undistort_device(const uint8_t* d_src, uint8_t* d_dst, int n, int W, int H, const double* K, const double* dist8, cudaStream_t stream,
                                    double** ir_buf = nullptr, size_t* ir_count = nullptr);
}

// Everything the launches of one VC_EXACT carve depend on: when it is unchanged, the captured CUDA graph of the last such
// carve (memset of the counters + the three kernels + the mid-point event) is launched again - one driver call instead of
// five, and no host-side launch gaps between kernels that run for tens of microseconds each.
struct CarveGraphKey {
    VcCarveParams p;
    const void* ptrs[10];
    int fresh, sm_count;
};
struct CarveGraphSlot {
    cudaGraphExec_t exec = nullptr;
    CarveGraphKey key;
    bool valid = false;
};

struct vc_engine {
    vc_grid_desc g{};
    int Wx = 0, nz = 0;
    unsigned long long uid = 0;
    long long slab_words = 0, plane_words = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evm = nullptr;
    cudaStream_t copy_stream = nullptr;   // D2H of finished z-chunks while the next chunk is carving (vc_carve_download)
    cudaStream_t fill_stream = nullptr;   // vc_blind_fill_kernel of a fresh carve, next to the brick classification
    cudaEvent_t ev_fill_fork = nullptr, ev_fill_join = nullptr;
    cudaEvent_t ev_chunk[4] = {nullptr, nullptr, nullptr, nullptr};
    bool have_mid = false;
    // volumes
    uint32_t *d_occ_own = nullptr, *d_seen_own = nullptr;    // slab-sized, engine-owned
    uint32_t *d_occ_full = nullptr, *d_seen_full = nullptr;  // whole grid: caller-owned (vc_bind_volumes) or the two below
    uint32_t *d_occ_full_own = nullptr, *d_seen_full_own = nullptr;  // vc_alloc_full_volumes
    bool gathered = false;
    // Halo planes of `occupied`: z_begin - 1 and z_end sit right next to the slab - inside the whole-grid buffer when one is
    // bound, in the two extra planes of d_occ_own otherwise - so the consumers address them like any other plane.
    bool halo_lo = false, halo_hi = false;   // valid (imported since the neighbour slab was last carved)
    cudaEvent_t ev_halo = nullptr;           // "my slab is complete" for vc_exchange_halos_peer
    ncclComm_t comm = nullptr;               // vc_comm_init
    int comm_rank = 0, comm_world = 1;
    unsigned long long* d_reduce = nullptr;  // staging of vc_comm_allreduce_u64
    size_t reduce_cap = 0;
    // views
    int V = 0, W = 0, H = 0, Ww = 0;
    unsigned long long views_version = 0;
    std::vector<VcViewConst> h_view;
    std::vector<float> h_cam;
    std::vector<VcViewFilter> h_filt;
    float hDu = 0.f, hDv = 0.f;          // thresholds of the per-voxel filter (vc_filter_constants)
    bool have_M = false;
    uint32_t* d_mask = nullptr;
    VcViewFilter* d_filt = nullptr;      // global copy of c_filt for lane-divergent reads (sub-brick classification)
    VcViewConst* d_view64 = nullptr;     // global copy of c_view for lane-divergent reads (deferred exact evaluations)
    float4* d_cam = nullptr;             // camera translations of all V views when V > VC_MAX_VIEWS (the colour pass over every group)
    vc_sat_t* d_sat = nullptr;           // summed-area tables of the background bits modulo 2^16, V x (H+1) x (W+1)
    uint32_t* d_sat_tmp = nullptr;       // V x H x Ww word-column prefixes used while building d_sat
    uint8_t* d_bgr_tmp = nullptr;        // staging for 8UC3 masks (grow-only)
    size_t bgr_tmp_bytes = 0;
    VcBrickState* d_bricks = nullptr;    // work list: bricks of the slab that need per-voxel evaluation
    VcBrickState* d_super = nullptr;     // dense states of the super-bricks (level 1 of the classifier)
    uint8_t* d_brick_flags = nullptr;    // VC_BRICK_* flags per brick
    uint8_t* d_super_flags = nullptr;    // ... per super-brick
    unsigned int* d_super_list = nullptr;
    CarveGraphSlot graph_slot[2];        // [fresh] cached graphs of a whole-range VC_EXACT carve
    int use_graphs = -1;                 // -1: not decided yet (environment variable VOXCARVE_NO_GRAPH=1 switches them off)
    bool profiling = false;              // vc_set_profiling: plain launches with an event between classification and per-voxel kernel
    int resident_blocks = 0;             // of vc_carve_bricks per SM (occupancy query, once)
    bool reset_pending = false;          // vc_reset not yet materialised (a VC_EXACT carve folds it into its fill pass)
    bool flags_valid = false;            // the brick / super-brick flags describe the volumes as they are (after a fresh whole-range VC_EXACT carve)
    bool carved_implies_seen = true;     // invariant of every state the engine produces; uploaded volumes may break it (vc_upload_volumes)
    // grow-only scratch shared by vc_fast_carve (flood volume), vc_mc_mesh (column counts), vc_mesh_from_volumes (column counts,
    // record row table, dilated occupancy), raw uploads and the
    // carved-but-unseen path of vc_carve: none of them runs concurrently with another on this engine's stream
    uint32_t *d_sparse_idx = nullptr, *d_sparse_words = nullptr;  // vc_carve_download_sparse (grow-only)
    unsigned long long sparse_cap = 0;
    void* d_scratch = nullptr;
    size_t scratch_bytes = 0;
    double* d_undist_ir = nullptr;       // per-stripe inverse camera matrices and row block starts of the device cv::undistort (grow-only)
    size_t undist_ir_count = 0;
    int sm_count = 148;
    uint8_t* d_images = nullptr;
    size_t mask_bytes = 0;
    // colour / mc results
    unsigned long long *d_block_sums = nullptr, *d_scalars = nullptr;  // scalars: [2]=executed, [3..4]=popcounts, [5]=corner projections, [6]=work-list front | super-list lengths, [7]=work counter | work-list back length, [8..11]=filter statistics
    unsigned long long* d_color_idx = nullptr;
    uchar4* d_color_rgbn = nullptr;
    unsigned long long n_surface = 0, color_capacity = 0;  // colour record buffers are grow-only
    bool have_colors = false;
    unsigned long long* d_hist = nullptr;
    bool have_mc = false;
    // dense RGBA model ("next" rows)
    float4 *d_dense = nullptr, *d_dense_tmp = nullptr;
    float* d_mesh_verts = nullptr;
    uint32_t* d_mesh_rgb = nullptr;
    unsigned long long n_mesh_tris = 0, mesh_capacity = 0;
    bool have_dense = false, have_mesh = false;
    unsigned long long mesh_version = 0;  // bumped whenever the mesh buffers are rewritten or freed
    // .off text of the mesh (vc_mesh_format_off), grow-only; valid while mesh_version == text_version
    char* d_text = nullptr;
    unsigned long long text_capacity = 0, text_bytes = 0, text_version = 0;
    bool have_text = false;
    bool have_calib = false;
    double calib_K[9] = {0}, calib_dist[8] = {0};
    vc_stats stats{};
    std::string err;

    uint32_t* occ_slab() const { return d_occ_full ? d_occ_full + (long long)g.z_begin * plane_words : d_occ_own + plane_words; }  // own: one halo plane in front
    uint32_t* seen_slab() const { return d_seen_full ? d_seen_full + (long long)g.z_begin * plane_words : d_seen_own; }
    bool whole_grid() const { return g.z_begin == 0 && g.z_end == g.Z; }
};

namespace {

int fail(vc_engine* e, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (e) e->err = buf; else g_create_error = buf;
    return code;
}

#define VC_CUDA(e, call)                                                                              \
    do {                                                                                              \
        cudaError_t _s = (call);                                                                      \
        if (_s != cudaSuccess)                                                                        \
            return fail((e), VC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_s), __FILE__, __LINE__); \
    } while (0)

int bind_device(vc_engine* e) {
    VC_CUDA(e, cudaSetDevice(e->g.device));
    return VC_OK;
}

// grow-only scratch; the caller owns it until its work on e->stream is enqueued (stream order protects the next user)
int ensure_scratch(vc_engine* e, size_t bytes, void** out) {
    if (e->scratch_bytes < bytes) {
        VC_CUDA(e, cudaStreamSynchronize(e->stream));
        cudaFree(e->d_scratch); e->d_scratch = nullptr; e->scratch_bytes = 0;
        VC_CUDA(e, cudaMalloc(&e->d_scratch, bytes));
        e->scratch_bytes = bytes;
    }
    *out = e->d_scratch;
    return VC_OK;
}

bool host_pinned(const void* p) {  // page-locked (cudaHostAlloc / cudaHostRegister) host memory?
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// ---------------------------------------------------------------------------------------------
// Volume memory.  The occupancy / seen volumes are written once per carve, almost entirely with uniform words (all occupied,
// all carved, all seen), and read again by every consumer.  They live in COMPRESSIBLE device memory when the GPU grants it
// (cuMemCreate + CU_MEM_ALLOCATION_COMP_GENERIC: the L2 compresses uniform lines on their way to HBM), plain cudaMalloc memory
// otherwise or with VOXCARVE_COMPRESSIBLE=0.  The driver entry points come from cudaGetDriverEntryPoint: no link against libcuda.
// ---------------------------------------------------------------------------------------------
struct VmmApi {
    bool tried = false, ok = false;
    CUresult (*MemCreate)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
    CUresult (*MemRelease)(CUmemGenericAllocationHandle) = nullptr;
    CUresult (*MemAddressReserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*MemAddressFree)(CUdeviceptr, size_t) = nullptr;
    CUresult (*MemMap)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
    CUresult (*MemUnmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*MemSetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
    CUresult (*MemGetAllocationGranularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
    CUresult (*MemGetAllocationPropertiesFromHandle)(CUmemAllocationProp*, CUmemGenericAllocationHandle) = nullptr;
    CUresult (*DeviceGetAttribute)(int*, CUdevice_attribute, CUdevice) = nullptr;
    CUresult (*DevicePrimaryCtxGetState)(CUdevice, unsigned int*, int*) = nullptr;
};
struct VmmBlock { size_t size; CUmemGenericAllocationHandle handle; unsigned long long access_mask; };  // bit d: device d may read / write it
static VmmApi g_vmm;
static std::mutex g_vmm_mutex;
static std::map<void*, VmmBlock> g_vmm_blocks;

static bool vmm_load() {  // g_vmm_mutex held
    if (g_vmm.tried) return g_vmm.ok;
    g_vmm.tried = true;
    const char* env = getenv("VOXCARVE_COMPRESSIBLE");
    if (env && env[0] == '0') return false;
    bool ok = true;
    auto get = [&](const char* name, void** fn) {
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !*fn) { cudaGetLastError(); ok = false; }
    };
    get("cuMemCreate", (void**)&g_vmm.MemCreate);
    get("cuMemRelease", (void**)&g_vmm.MemRelease);
    get("cuMemAddressReserve", (void**)&g_vmm.MemAddressReserve);
    get("cuMemAddressFree", (void**)&g_vmm.MemAddressFree);
    get("cuMemMap", (void**)&g_vmm.MemMap);
    get("cuMemUnmap", (void**)&g_vmm.MemUnmap);
    get("cuMemSetAccess", (void**)&g_vmm.MemSetAccess);
    get("cuMemGetAllocationGranularity", (void**)&g_vmm.MemGetAllocationGranularity);
    get("cuMemGetAllocationPropertiesFromHandle", (void**)&g_vmm.MemGetAllocationPropertiesFromHandle);
    get("cuDeviceGetAttribute", (void**)&g_vmm.DeviceGetAttribute);
    get("cuDevicePrimaryCtxGetState", (void**)&g_vmm.DevicePrimaryCtxGetState);
    g_vmm.ok = ok;
    return ok;
}

// compressible memory on `device` (the current one), readable / writable from the devices this process already works on and can
// reach it from (the other engines of a multi-engine host; a process per GPU maps its own device only); engines that come later
// are granted access when they first take part in a peer copy (vol_grant_access); nullptr = not granted
static void* vmm_alloc_compressible(int device, size_t bytes) {
    std::lock_guard<std::mutex> lk(g_vmm_mutex);
    if (!vmm_load()) return nullptr;
    int supported = 0;
    if (g_vmm.DeviceGetAttribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, (CUdevice)device) != CUDA_SUCCESS || !supported) return nullptr;
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    if (g_vmm.MemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0) return nullptr;
    const size_t size = (bytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle h;
    if (g_vmm.MemCreate(&h, size, &prop, 0) != CUDA_SUCCESS) return nullptr;
    CUmemAllocationProp got = {};
    if (g_vmm.MemGetAllocationPropertiesFromHandle(&got, h) != CUDA_SUCCESS || got.allocFlags.compressionType != CU_MEM_ALLOCATION_COMP_GENERIC) { g_vmm.MemRelease(h); return nullptr; }
    CUdeviceptr va = 0;
    if (g_vmm.MemAddressReserve(&va, size, 0, 0, 0) != CUDA_SUCCESS) { g_vmm.MemRelease(h); return nullptr; }
    if (g_vmm.MemMap(va, size, 0, h, 0) != CUDA_SUCCESS) { g_vmm.MemAddressFree(va, size); g_vmm.MemRelease(h); return nullptr; }
    std::vector<CUmemAccessDesc> acc;
    unsigned long long mask = 0;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess) { cudaGetLastError(); n_dev = device + 1; }
    for (int d = 0; d < n_dev && d < 64; d++) {  // the halo / gather copies between engines of one process read and write peers' volumes
        int can = d == device;
        if (!can) {
            unsigned int flags = 0;
            int active = 0;
            if (g_vmm.DevicePrimaryCtxGetState((CUdevice)d, &flags, &active) != CUDA_SUCCESS || !active) continue;  // not a device of this process (so far)
            if (cudaDeviceCanAccessPeer(&can, d, device) != cudaSuccess) { cudaGetLastError(); can = 0; }
        }
        if (!can) continue;
        CUmemAccessDesc a = {};
        a.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
        a.location.id = d;
        a.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        acc.push_back(a);
        mask |= 1ull << d;
    }
    if (g_vmm.MemSetAccess(va, size, acc.data(), acc.size()) != CUDA_SUCCESS) {
        CUmemAccessDesc a = {};  // at least the owner
        a.location.type = CU_MEM_LOCATION_TYPE_DEVICE; a.location.id = device; a.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        mask = 1ull << device;
        if (g_vmm.MemSetAccess(va, size, &a, 1) != CUDA_SUCCESS) { g_vmm.MemUnmap(va, size); g_vmm.MemAddressFree(va, size); g_vmm.MemRelease(h); return nullptr; }
    }
    g_vmm_blocks[(void*)va] = VmmBlock{size, h, mask};
    return (void*)va;
}

// before a copy between engines: let `device` read / write the volume that holds address `p` (no-op for cudaMalloc / caller memory)
static void vol_grant_access(const void* p, int device) {
    if (!p || device < 0 || device >= 64) return;
    std::lock_guard<std::mutex> lk(g_vmm_mutex);
    auto it = g_vmm_blocks.upper_bound((void*)p);  // first block that starts beyond p
    if (it == g_vmm_blocks.begin()) return;
    --it;
    if ((const char*)p >= (const char*)it->first + it->second.size || (it->second.access_mask >> device) & 1ull) return;
    CUmemAccessDesc a = {};
    a.location.type = CU_MEM_LOCATION_TYPE_DEVICE; a.location.id = device; a.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (g_vmm.MemSetAccess((CUdeviceptr)it->first, it->second.size, &a, 1) == CUDA_SUCCESS) it->second.access_mask |= 1ull << device;
}
static void grant_peer_access(vc_engine* owner, int device) {  // all of `owner`'s engine-owned volumes
    vol_grant_access(owner->d_occ_own, device); vol_grant_access(owner->d_seen_own, device);
    vol_grant_access(owner->d_occ_full_own, device); vol_grant_access(owner->d_seen_full_own, device);
}

static cudaError_t vol_alloc(vc_engine* e, uint32_t** out, size_t bytes) {
    *out = (uint32_t*)vmm_alloc_compressible(e->g.device, bytes);
    if (*out) { e->stats.volumes_compressible = 1; return cudaSuccess; }
    e->stats.volumes_compressible = 0;
    return cudaMalloc(out, bytes);
}
static void vol_free(uint32_t* p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(g_vmm_mutex);
        auto it = g_vmm_blocks.find((void*)p);
        if (it != g_vmm_blocks.end()) {
            cudaDeviceSynchronize();  // cudaFree's implicit wait for work in flight, restated
            g_vmm.MemUnmap((CUdeviceptr)p, it->second.size);
            g_vmm.MemAddressFree((CUdeviceptr)p, it->second.size);
            g_vmm.MemRelease(it->second.handle);
            g_vmm_blocks.erase(it);
            return;
        }
    }
    cudaFree(p);
}

// Views come in groups of VC_MAX_VIEWS consecutive views, group g = views [g * VC_MAX_VIEWS, (g + 1) * VC_MAX_VIEWS); the
// constant tables hold one group at a time.  An engine with at most VC_MAX_VIEWS views has one group and uploads it once.
int n_groups(const vc_engine* e) { return (e->V + VC_MAX_VIEWS - 1) / VC_MAX_VIEWS; }

// upload view group `group` of this engine to the constant tables if another engine (or another version or group) owns them
int ensure_constants(vc_engine* e, int group = 0) {
    std::lock_guard<std::mutex> lk(g_const_mutex);
    ConstOwner& o = g_const_owner[e->g.device & 63];
    if (o.uid == e->uid && o.version == e->views_version && o.group == group) return VC_OK;
    // c_view / c_cam / c_filt are per-device symbols shared by every engine on this GPU: kernels of the previous owner (another
    // engine, or this one with older views) may still be reading them on another stream.  This engine's own kernels of another
    // group run on e->stream, ahead of the copies below, so switching groups inside one call needs no host synchronisation.
    if (o.used && o.last_use && (o.uid != e->uid || e->V <= VC_MAX_VIEWS)) VC_CUDA(e, cudaEventSynchronize(o.last_use));
    o.used = false;
    const int v0 = group * VC_MAX_VIEWS, nv = std::min(VC_MAX_VIEWS, e->V - v0);
    VC_CUDA(e, cudaMemcpyToSymbolAsync(c_view, e->h_view.data() + v0, sizeof(VcViewConst) * nv, 0, cudaMemcpyHostToDevice, e->stream));
    VC_CUDA(e, cudaMemcpyToSymbolAsync(c_cam, e->h_cam.data() + (size_t)v0 * 4, sizeof(float) * 4 * nv, 0, cudaMemcpyHostToDevice, e->stream));
    VC_CUDA(e, cudaMemcpyToSymbolAsync(c_filt, e->h_filt.data() + v0, sizeof(VcViewFilter) * nv, 0, cudaMemcpyHostToDevice, e->stream));
    // the host vectors may change right after this call returns; make the copy complete first.  (With several groups they
    // cannot: vc_set_views and vc_append_views synchronise the stream before they touch them.)
    if (e->V <= VC_MAX_VIEWS) VC_CUDA(e, cudaStreamSynchronize(e->stream));
    o.uid = e->uid;
    o.version = e->views_version;
    o.group = group;
    return VC_OK;
}

// call after the last launch of an entry point that reads the view constants
int constants_used(vc_engine* e) {
    std::lock_guard<std::mutex> lk(g_const_mutex);
    ConstOwner& o = g_const_owner[e->g.device & 63];
    if (o.uid != e->uid) return VC_OK;
    if (!o.last_use) VC_CUDA(e, cudaEventCreateWithFlags(&o.last_use, cudaEventDisableTiming));
    VC_CUDA(e, cudaEventRecord(o.last_use, e->stream));
    o.used = true;
    return VC_OK;
}

// planes of the occupancy volume that kernels may address: [cz0, cz1) starting at `base`
VcVolView vol_view(const vc_engine* e) {
    VcVolView g;
    g.X = e->g.X; g.Y = e->g.Y; g.Z = e->g.Z; g.Wx = e->Wx;
    if (e->d_occ_full && e->gathered) { g.base = e->d_occ_full; g.cz0 = 0; g.cz1 = e->g.Z; }
    else {
        const int lo = (e->halo_lo && e->g.z_begin > 0) ? 1 : 0, hi = (e->halo_hi && e->g.z_end < e->g.Z) ? 1 : 0;
        g.base = e->occ_slab() - (long long)lo * e->plane_words; g.cz0 = e->g.z_begin - lo; g.cz1 = e->g.z_end + hi;
    }
    return g;
}

// launch with programmatic stream serialization: the kernel may begin while the previous kernel of the stream drains (it
// synchronises itself with vc_pdl_wait before touching that kernel's results)
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t stream, bool pdl, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

template <int K>
int launch_carve(vc_engine* e, int mode, const VcCarveParams& p, bool count) {
    const long long blocks = (long long)p.G * p.YB * e->nz;
    if (blocks > 0x7fffffffLL) return fail(e, VC_ERR_ARG, "slab too large for one launch (%lld blocks)", blocks);
    dim3 grid((unsigned)blocks), block(32 * VC_TILE_ROWS);
    if (mode == VC_EXACT) {
        if (count) vc_carve_rows<K, true, true><<<grid, block, 0, e->stream>>>(p);
        else vc_carve_rows<K, true, false><<<grid, block, 0, e->stream>>>(p);
    } else {
        if (count) vc_carve_rows<K, false, true><<<grid, block, 0, e->stream>>>(p);
        else vc_carve_rows<K, false, false><<<grid, block, 0, e->stream>>>(p);
    }
    VC_CUDA(e, cudaGetLastError());
    e->stats.carve_launches++;
    return VC_OK;
}

void free_color(vc_engine* e) {
    cudaFree(e->d_color_idx); e->d_color_idx = nullptr;
    cudaFree(e->d_color_rgbn); e->d_color_rgbn = nullptr;
    e->color_capacity = 0;
    e->have_colors = false;
    e->n_surface = 0;
}

// Error-radius coefficients of the per-voxel f32 filter (derivation above vc_filter_coord in vc_kernels.cuh), in f64 with
// every factor rounded up.  T_i bounds sum_k |P_ik w_k| over the WHOLE grid (any slab of it), w = (y s, x s, -z s, 1) as f32
// products.  A view whose matrix is not finite, or so large that the f32 evaluation could overflow, gets Cu = Cv = +inf:
// its voxel-views are then never "decided" and all go through the exact path.
void vc_filter_constants(vc_engine* e, VcViewFilter* filt, int n) {
    const double up = 1.0 + ldexp(1.0, -22);  // f32 rounding of the coordinate products, with room to spare
    const double s = (double)e->g.voxel_size;
    const double ax = (double)(e->g.X - 1) * s * up, ay = (double)(e->g.Y - 1) * s * up, az = (double)(e->g.Z - 1) * s * up;
    const double W3 = (double)e->W + 3.0, H3 = (double)e->H + 3.0;
    for (int v = 0; v < n; v++) {
        VcViewFilter& f = filt[v];
        double eta[3];
        bool ok = true;
        for (int i = 0; i < 3; i++) {
            const double T = fabs((double)f.P[i * 4 + 0]) * ay + fabs((double)f.P[i * 4 + 1]) * ax + fabs((double)f.P[i * 4 + 2]) * az + fabs((double)f.P[i * 4 + 3]);
            ok = ok && std::isfinite(T) && T < ldexp(1.0, 60);
            eta[i] = 4.0 * ldexp(1.0, -24) * T * (1.0 + ldexp(1.0, -19)) + ldexp(1.0, -100);
        }
        const double Cu = (eta[0] + W3 * eta[2]) * (1.0 + ldexp(1.0, -19)), Cv = (eta[1] + H3 * eta[2]) * (1.0 + ldexp(1.0, -19));
        f.Cu = ok ? nextafterf((float)Cu, INFINITY) : INFINITY;
        f.Cv = ok ? nextafterf((float)Cv, INFINITY) : INFINITY;
        f.pad[0] = f.pad[1] = 0.0f;
    }
    const double Du = W3 * ldexp(1.0, -22) * (1.0 + ldexp(1.0, -10)) + ldexp(1.0, -20);
    const double Dv = H3 * ldexp(1.0, -22) * (1.0 + ldexp(1.0, -10)) + ldexp(1.0, -20);
    e->hDu = nextafterf((float)(0.5 - Du), -INFINITY);
    e->hDv = nextafterf((float)(0.5 - Dv), -INFINITY);
}

}  // namespace

extern "C" {

int vc_api_version(void) { return VC_API_VERSION; }

const char* vc_last_error(const vc_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int vc_create(const vc_grid_desc* grid, vc_engine** out) {
    if (!grid || !out) return fail(nullptr, VC_ERR_ARG, "vc_create: null argument");
    *out = nullptr;
    const vc_grid_desc& g = *grid;
    // main.cpp:232-246: x, y, z >= 1 and size > 0
    if (g.X < 1 || g.Y < 1 || g.Z < 1) return fail(nullptr, VC_ERR_ARG, "vc_create: grid dims must be >= 1 (got %d %d %d)", g.X, g.Y, g.Z);
    if (!(g.voxel_size > 0.0f)) return fail(nullptr, VC_ERR_ARG, "vc_create: voxel size must be strictly positive");
    if (g.z_begin < 0 || g.z_end > g.Z || g.z_begin >= g.z_end)
        return fail(nullptr, VC_ERR_ARG, "vc_create: bad z-slab [%d,%d) for Z=%d", g.z_begin, g.z_end, g.Z);
    int ndev = 0;
    cudaError_t s = cudaGetDeviceCount(&ndev);
    if (s != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, VC_ERR_CUDA, "vc_create: no CUDA device (%s); this engine has no CPU fallback",
                    s != cudaSuccess ? cudaGetErrorString(s) : "device count 0");
    }
    if (g.device < 0 || g.device >= ndev) return fail(nullptr, VC_ERR_ARG, "vc_create: device %d out of range (%d devices)", g.device, ndev);
    vc_engine* e = new vc_engine();
    e->g = g;
    e->Wx = (g.X + 31) / 32;
    e->nz = g.z_end - g.z_begin;
    e->plane_words = (long long)g.Y * e->Wx;
    e->slab_words = e->plane_words * e->nz;
    {
        std::lock_guard<std::mutex> lk(g_const_mutex);
        e->uid = g_next_uid++;
    }
#define VC_CREATE_CUDA(call)                                                                   \
    do {                                                                                       \
        cudaError_t _s = (call);                                                               \
        if (_s != cudaSuccess) {                                                               \
            fail(nullptr, VC_ERR_CUDA, "vc_create: %s failed: %s", #call, cudaGetErrorString(_s)); \
            vc_destroy(e);                                                                     \
            return VC_ERR_CUDA;                                                                \
        }                                                                                      \
    } while (0)
    VC_CREATE_CUDA(cudaSetDevice(g.device));
    VC_CREATE_CUDA(cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, g.device));
    VC_CREATE_CUDA(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
    e->stream = e->own_stream;
    VC_CREATE_CUDA(cudaEventCreate(&e->ev0));
    VC_CREATE_CUDA(cudaEventCreate(&e->ev1));
    VC_CREATE_CUDA(cudaEventCreate(&e->evm));
    VC_CREATE_CUDA(cudaMalloc(&e->d_scalars, 16 * sizeof(unsigned long long)));
    VC_CREATE_CUDA(cudaMalloc(&e->d_hist, 257 * sizeof(unsigned long long)));  // [256] = task counter of vc_mc_classify_kernel
    VC_CREATE_CUDA(cudaMalloc(&e->d_filt, VC_MAX_VIEWS * sizeof(VcViewFilter)));
    VC_CREATE_CUDA(cudaMalloc(&e->d_view64, VC_MAX_VIEWS * sizeof(VcViewConst)));
#undef VC_CREATE_CUDA
    *out = e;
    int rc = vc_reset(e);
    if (rc != VC_OK) { g_create_error = e->err; vc_destroy(e); *out = nullptr; return rc; }
    return VC_OK;
}

void vc_destroy(vc_engine* e) {
    if (!e) return;
    cudaSetDevice(e->g.device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    vol_free(e->d_occ_own); vol_free(e->d_seen_own); cudaFree(e->d_mask); cudaFree(e->d_images);
    cudaFree(e->d_sat); cudaFree(e->d_sat_tmp); cudaFree(e->d_bgr_tmp); cudaFree(e->d_bricks); cudaFree(e->d_super); cudaFree(e->d_brick_flags); cudaFree(e->d_super_flags); cudaFree(e->d_super_list);
    cudaFree(e->d_block_sums);
    cudaFree(e->d_scalars); cudaFree(e->d_hist); cudaFree(e->d_filt); cudaFree(e->d_view64); cudaFree(e->d_cam);
    cudaFree(e->d_dense); cudaFree(e->d_dense_tmp); cudaFree(e->d_mesh_verts); cudaFree(e->d_mesh_rgb); cudaFree(e->d_text);
    cudaFree(e->d_sparse_idx); cudaFree(e->d_sparse_words);
    cudaFree(e->d_scratch); cudaFree(e->d_undist_ir); vol_free(e->d_occ_full_own); vol_free(e->d_seen_full_own); cudaFree(e->d_reduce);
    if (e->comm) vc_comm_destroy(e);
    for (CarveGraphSlot& gs : e->graph_slot) if (gs.exec) cudaGraphExecDestroy(gs.exec);
    if (e->ev_halo) cudaEventDestroy(e->ev_halo);
    free_color(e);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->evm) cudaEventDestroy(e->evm);
    for (int c = 0; c < 4; c++) if (e->ev_chunk[c]) cudaEventDestroy(e->ev_chunk[c]);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->ev_fill_fork) cudaEventDestroy(e->ev_fill_fork);
    if (e->ev_fill_join) cudaEventDestroy(e->ev_fill_join);
    if (e->fill_stream) cudaStreamDestroy(e->fill_stream);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    {
        std::lock_guard<std::mutex> lk(g_const_mutex);
        ConstOwner& o = g_const_owner[e->g.device & 63];
        if (o.uid == e->uid) { o.uid = 0; o.version = 0; o.group = 0; o.used = false; }  // the stream was synchronised above; the event is kept for the device
    }
    delete e;
}

int vc_set_stream(vc_engine* e, void* cuda_stream) {
    if (!e) return VC_ERR_ARG;
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
    return VC_OK;
}

int vc_set_profiling(vc_engine* e, int32_t on) {
    if (!e) return VC_ERR_ARG;
    e->profiling = on != 0;
    return VC_OK;
}

int vc_synchronize(vc_engine* e) {
    if (!e) return VC_ERR_ARG;
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

int vc_set_views(vc_engine* e, int32_t V, int32_t W, int32_t H, const float* P, const float* M) {
    if (!e) return VC_ERR_ARG;
    if (!P) return fail(e, VC_ERR_ARG, "vc_set_views: P is null");
    if (V < 1 || V > VC_MAX_VIEWS) return fail(e, VC_ERR_ARG, "vc_set_views: V=%d outside [1,%d]", V, VC_MAX_VIEWS);
    if (W < 1 || H < 1 || W > (1 << 20) || H > (1 << 20)) return fail(e, VC_ERR_ARG, "vc_set_views: image size %dx%d outside [1,2^20]", W, H);
    // every check before any state changes: a refused call leaves the engine's views, masks, tables and images as they were
    const int Ww = (W + 31) / 32;
    const size_t mask_bytes = (size_t)V * H * Ww * 4;
    if ((unsigned long long)vc_sat_pitch(W) * (H + 1) > 0x7fffffffull) return fail(e, VC_ERR_ARG, "vc_set_views: image %dx%d too large for 32-bit SAT offsets", W, H);
    if (mask_bytes / 4 > 0x7fffffffull) return fail(e, VC_ERR_ARG, "vc_set_views: %d views of %dx%d exceed 2^31 mask words", V, W, H);
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    if (V != e->V || W != e->W || H != e->H) {  // geometry changed: masks / images no longer match
        cudaFree(e->d_mask); e->d_mask = nullptr;
        cudaFree(e->d_sat); e->d_sat = nullptr;
        cudaFree(e->d_sat_tmp); e->d_sat_tmp = nullptr;
        cudaFree(e->d_images); e->d_images = nullptr;
    }
    e->V = V; e->W = W; e->H = H; e->Ww = Ww;
    e->mask_bytes = mask_bytes;
    e->h_view.resize(V);
    e->h_cam.assign((size_t)V * 4, 0.0f);
    e->h_filt.assign((size_t)V, VcViewFilter{});
    for (int v = 0; v < V; v++) {
        for (int k = 0; k < 12; k++) e->h_view[v].P[k] = (double)P[v * 12 + k];
        for (int k = 0; k < 12; k++) e->h_filt[v].P[k] = P[v * 12 + k];
        if (M) {
            e->h_cam[v * 4 + 0] = M[v * 12 + 3];
            e->h_cam[v * 4 + 1] = M[v * 12 + 7];
            e->h_cam[v * 4 + 2] = M[v * 12 + 11];
            e->h_cam[v * 4 + 3] = 1.0f;
        }
    }
    e->have_M = M != nullptr;
    vc_filter_constants(e, e->h_filt.data(), V);
    VC_CUDA(e, cudaMemcpyAsync(e->d_filt, e->h_filt.data(), sizeof(VcViewFilter) * V, cudaMemcpyHostToDevice, e->stream));  // h_filt lives until the next vc_set_views, which synchronises first
    VC_CUDA(e, cudaMemcpyAsync(e->d_view64, e->h_view.data(), sizeof(VcViewConst) * V, cudaMemcpyHostToDevice, e->stream));
    e->views_version++;
    return VC_OK;
}

// bit packing (8UC3 input: bgr = the pixels of view v0, else nullptr) and summed-area tables of the views [v0, v1) into the
// given mask / table buffers, on the engine's stream
static cudaError_t build_view_tables(vc_engine* e, const uint8_t* bgr, uint32_t* mask, uint32_t* sat_tmp, vc_sat_t* sat, int v0, int v1) {
    const size_t view_words = (size_t)e->H * e->Ww;
    const int nv = v1 - v0;
    uint32_t* m = mask + (size_t)v0 * view_words;
    uint32_t* t = sat_tmp + (size_t)v0 * view_words;
    const long long n_rows = (long long)nv * e->H;
    const int n_cols = nv * e->Ww;
    if (bgr) {
        const long long warps = n_rows * e->Ww;
        vc_pack_bgr_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, e->stream>>>(bgr, m, e->W, e->Ww, n_rows);
    }
    vc_sat_rowprefix_kernel<<<(unsigned)((n_rows + 7) / 8), 256, 0, e->stream>>>(m, t, e->Ww, n_rows);  // a warp per row
    vc_sat_build_kernel<<<(unsigned)n_cols, 32 * VC_SAT_WARPS, 0, e->stream>>>(m, t, sat + (size_t)v0 * (e->H + 1) * vc_sat_pitch(e->W), e->W, e->H, e->Ww, nv);
    return cudaGetLastError();
}

int vc_set_masks(vc_engine* e, const void* masks, int32_t format) {
    if (!e) return VC_ERR_ARG;
    if (!masks) return fail(e, VC_ERR_ARG, "vc_set_masks: null buffer");
    if (e->V == 0) return fail(e, VC_ERR_STATE, "vc_set_masks: call vc_set_views first");
    if (format != VC_MASK_BITS && format != VC_MASK_BGR8 && format != VC_MASK_BGR8_RAW) return fail(e, VC_ERR_ARG, "vc_set_masks: unknown format %d", format);
    if (format == VC_MASK_BGR8_RAW && !e->have_calib) return fail(e, VC_ERR_STATE, "vc_set_masks: raw masks need vc_set_calibration first");
    if (format == VC_MASK_BGR8_RAW && (e->W > VC_RAW_MAX_SIDE || e->H > VC_RAW_MAX_SIDE))
        return fail(e, VC_ERR_ARG, "vc_set_masks: raw masks of %dx%d: cv::undistort takes W and H up to %d", e->W, e->H, VC_RAW_MAX_SIDE);
    if (bind_device(e)) return VC_ERR_CUDA;
    if (!e->d_mask) VC_CUDA(e, cudaMalloc(&e->d_mask, e->mask_bytes));
    const size_t sat_words = (size_t)e->V * (e->H + 1) * vc_sat_pitch(e->W);
    if (!e->d_sat) VC_CUDA(e, cudaMalloc(&e->d_sat, sat_words * sizeof(vc_sat_t)));
    if (!e->d_sat_tmp) VC_CUDA(e, cudaMalloc(&e->d_sat_tmp, e->mask_bytes));
    const size_t view_bgr = (size_t)e->H * e->W * 3;
    const size_t bgr_bytes = (size_t)e->V * view_bgr;
    uint8_t* d_tmp = nullptr;
    if (format != VC_MASK_BITS) {
        if (e->bgr_tmp_bytes < bgr_bytes) {
            VC_CUDA(e, cudaStreamSynchronize(e->stream));
            cudaFree(e->d_bgr_tmp); e->d_bgr_tmp = nullptr; e->bgr_tmp_bytes = 0;
            VC_CUDA(e, cudaMalloc(&e->d_bgr_tmp, bgr_bytes));
            e->bgr_tmp_bytes = bgr_bytes;
        }
        d_tmp = e->d_bgr_tmp;
    }
    // (Uploading the views in groups on a second stream, each group's tables built while the next one travels, was measured on
    // C4 with page-locked masks: 1.66 ms per end-to-end step instead of 1.45 ms - the 0.2 ms of overlap are less than what the
    // extra copies, events and 9 more launches cost the host.  One copy, one table build.)
    if (format == VC_MASK_BITS) {
        VC_CUDA(e, cudaMemcpyAsync(e->d_mask, masks, e->mask_bytes, cudaMemcpyDefault, e->stream));  // host or device memory
    } else {
        VC_CUDA(e, cudaMemcpyAsync(d_tmp, masks, bgr_bytes, cudaMemcpyHostToDevice, e->stream));
        if (format == VC_MASK_BGR8_RAW) {  // cv::undistort(mask, undist_mask, cameraMatrix, distCoeffs) (VoxelCarving.cpp:36)
            void* sc = nullptr;
            int rcs = ensure_scratch(e, bgr_bytes, &sc);
            if (rcs) return rcs;
            uint8_t* d_und = (uint8_t*)sc;
            cudaError_t us = undistort_device(d_tmp, d_und, e->V, e->W, e->H, e->calib_K, e->calib_dist, e->stream, &e->d_undist_ir, &e->undist_ir_count);
            if (us == cudaSuccess) us = cudaMemcpyAsync(d_tmp, d_und, bgr_bytes, cudaMemcpyDeviceToDevice, e->stream);
            if (us != cudaSuccess) return fail(e, VC_ERR_CUDA, "vc_set_masks: undistort failed: %s", cudaGetErrorString(us));
        }
    }
    VC_CUDA(e, build_view_tables(e, d_tmp, e->d_mask, e->d_sat_tmp, e->d_sat, 0, e->V));
    return VC_OK;
}

int vc_set_images(vc_engine* e, const uint8_t* images_bgr) {
    if (!e) return VC_ERR_ARG;
    if (!images_bgr) return fail(e, VC_ERR_ARG, "vc_set_images: null buffer");
    if (e->V == 0) return fail(e, VC_ERR_STATE, "vc_set_images: call vc_set_views first");
    if (bind_device(e)) return VC_ERR_CUDA;
    const size_t bytes = (size_t)e->V * e->H * e->W * 3;
    if (!e->d_images) VC_CUDA(e, cudaMalloc(&e->d_images, bytes));
    VC_CUDA(e, cudaMemcpyAsync(e->d_images, images_bgr, bytes, cudaMemcpyHostToDevice, e->stream));
    return VC_OK;
}

// 3x3 inverse as cv::invert(DECOMP_LU) computes it for n == 3: the adjugate times 1/det, all zeros when det == 0.  f64 with no
// FMA contraction (every product is rounded through a volatile), as OpenCV's core module is built for x86-64 without FMA.
static void inv3x3_cv(const double* S, double* t) {
    auto mul = [](double a, double b) { volatile double p = a * b; return (double)p; };
    auto cof = [&](int a, int b, int c, int d, int e, int f, int g, int h) { return mul(S[a * 3 + b], S[c * 3 + d]) - mul(S[e * 3 + f], S[g * 3 + h]); };
    double det = mul(S[0], cof(1, 1, 2, 2, 1, 2, 2, 1)) - mul(S[1], cof(1, 0, 2, 2, 1, 2, 2, 0));
    det = det + mul(S[2], cof(1, 0, 2, 1, 1, 1, 2, 0));
    if (det == 0) { for (int i = 0; i < 9; i++) t[i] = 0; return; }
    const double d = 1. / det;
    t[0] = mul(cof(1, 1, 2, 2, 1, 2, 2, 1), d); t[1] = mul(cof(0, 2, 2, 1, 0, 1, 2, 2), d); t[2] = mul(cof(0, 1, 1, 2, 0, 2, 1, 1), d);
    t[3] = mul(cof(1, 2, 2, 0, 1, 0, 2, 2), d); t[4] = mul(cof(0, 0, 2, 2, 0, 2, 2, 0), d); t[5] = mul(cof(0, 2, 1, 0, 0, 0, 1, 2), d);
    t[6] = mul(cof(1, 0, 2, 1, 1, 1, 2, 0), d); t[7] = mul(cof(0, 1, 2, 0, 0, 0, 2, 1), d); t[8] = mul(cof(0, 0, 1, 1, 0, 1, 1, 0), d);
}

// device-to-device cv::undistort of n 8UC3 images on `stream`; W and H must be below 32767 (the callers refuse larger)
// ir_buf / ir_count: optional grow-only device buffer (an engine's) for the per-stripe inverse matrices followed by the rows'
// block starts, in doubles; else allocated per call
static cudaError_t undistort_device(const uint8_t* d_src, uint8_t* d_dst, int n, int W, int H, const double* K, const double* dist8, cudaStream_t stream,
                                    double** ir_buf, size_t* ir_count) {
    if (W < 1 || H < 1 || W > VC_RAW_MAX_SIDE || H > VC_RAW_MAX_SIDE) return cudaErrorInvalidValue;
    int stripe = (1 << 12) / W;
    if (stripe < 1) stripe = 1;
    if (stripe > H) stripe = H;
    const int n_stripes = (H + stripe - 1) / stripe;
    std::vector<double> ir((size_t)n_stripes * 9);
    for (int sidx = 0; sidx < n_stripes; sidx++) {
        double Ar[9];
        memcpy(Ar, K, sizeof Ar);
        Ar[5] = K[5] - (double)(sidx * stripe);
        inv3x3_cv(Ar, &ir[(size_t)sidx * 9]);
    }
    const size_t n_doubles = ir.size() + (size_t)H * (W / 8 + 1) * 3;
    double* d_ir = nullptr;
    cudaError_t s = cudaSuccess;
    if (ir_buf && *ir_count >= n_doubles) d_ir = *ir_buf;
    else {
        s = cudaMalloc(&d_ir, n_doubles * sizeof(double));
        if (s != cudaSuccess) return s;
        if (ir_buf) {  // the old buffer may still be read by a kernel on this stream
            if (*ir_buf) { cudaStreamSynchronize(stream); cudaFree(*ir_buf); }
            *ir_buf = d_ir; *ir_count = n_doubles;
        }
    }
    s = cudaMemcpyAsync(d_ir, ir.data(), ir.size() * sizeof(double), cudaMemcpyHostToDevice, stream);
    if (s == cudaSuccess) s = cudaStreamSynchronize(stream);  // `ir` is a local
    if (s == cudaSuccess) {
        VcUndistortParams p{};
        p.src = d_src; p.dst = d_dst; p.ir = d_ir; p.starts = d_ir + ir.size(); p.W = W; p.H = H; p.n = n; p.stripe = stripe;
        p.fx = K[0]; p.fy = K[4]; p.u0 = K[2]; p.v0 = K[5];
        p.k1 = dist8[0]; p.k2 = dist8[1]; p.p1 = dist8[2]; p.p2 = dist8[3]; p.k3 = dist8[4]; p.k4 = dist8[5]; p.k5 = dist8[6]; p.k6 = dist8[7];
        vc_undistort_rows_kernel<<<(H + 127) / 128, 128, 0, stream>>>(p);
        vc_undistort_kernel<<<dim3((W + 255) / 256, H, n), 256, 0, stream>>>(p);
        s = cudaGetLastError();
        if (s == cudaSuccess) s = cudaStreamSynchronize(stream);
    }
    if (!ir_buf) cudaFree(d_ir);
    return s;
}

// engine-owned volumes are allocated on first use (a planning engine, vc_plan_slabs, never needs them)
static int ensure_volumes(vc_engine* e) {
    if (e->d_occ_full || e->d_occ_own) return VC_OK;
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, vol_alloc(e, &e->d_occ_own, (e->slab_words + 2 * e->plane_words) * 4));  // + the halo planes z_begin - 1 and z_end
    VC_CUDA(e, vol_alloc(e, &e->d_seen_own, e->slab_words * 4));
    return VC_OK;
}

// write the Model-constructor state now if a vc_reset is still pending (every reader / writer of the volumes calls this)
static int materialize_reset(vc_engine* e) {
    int rcv = ensure_volumes(e);
    if (rcv) return rcv;
    if (!e->reset_pending) return VC_OK;
    if (bind_device(e)) return VC_ERR_CUDA;
    const long long n = e->slab_words;
    vc_reset_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(e->occ_slab(), e->seen_slab(), n, e->Wx, e->g.X);
    VC_CUDA(e, cudaGetLastError());
    e->reset_pending = false;
    return VC_OK;
}

int vc_set_calibration(vc_engine* e, const double K[9], const double* dist, int32_t n_dist) {
    if (!e) return VC_ERR_ARG;
    if (!K || !dist) return fail(e, VC_ERR_ARG, "vc_set_calibration: null argument");
    if (n_dist != 4 && n_dist != 5 && n_dist != 8) return fail(e, VC_ERR_ARG, "vc_set_calibration: %d distortion coefficients (need 4, 5 or 8)", n_dist);
    for (int i = 0; i < 9; i++) e->calib_K[i] = K[i];
    for (int i = 0; i < 8; i++) e->calib_dist[i] = i < n_dist ? dist[i] : 0.0;
    e->have_calib = true;
    return VC_OK;
}

int vc_set_images_raw(vc_engine* e, const uint8_t* images_bgr) {
    if (!e) return VC_ERR_ARG;
    if (!images_bgr) return fail(e, VC_ERR_ARG, "vc_set_images_raw: null buffer");
    if (e->V == 0) return fail(e, VC_ERR_STATE, "vc_set_images_raw: call vc_set_views first");
    if (!e->have_calib) return fail(e, VC_ERR_STATE, "vc_set_images_raw: needs vc_set_calibration first");
    if (e->W > VC_RAW_MAX_SIDE || e->H > VC_RAW_MAX_SIDE)
        return fail(e, VC_ERR_ARG, "vc_set_images_raw: images of %dx%d: cv::undistort takes W and H up to %d", e->W, e->H, VC_RAW_MAX_SIDE);
    if (bind_device(e)) return VC_ERR_CUDA;
    const size_t bytes = (size_t)e->V * e->H * e->W * 3;
    if (!e->d_images) VC_CUDA(e, cudaMalloc(&e->d_images, bytes));
    void* sc = nullptr;
    int rcs = ensure_scratch(e, bytes, &sc);
    if (rcs) return rcs;
    uint8_t* d_raw = (uint8_t*)sc;
    cudaError_t s = cudaMemcpyAsync(d_raw, images_bgr, bytes, cudaMemcpyHostToDevice, e->stream);
    if (s == cudaSuccess) s = undistort_device(d_raw, e->d_images, e->V, e->W, e->H, e->calib_K, e->calib_dist, e->stream, &e->d_undist_ir, &e->undist_ir_count);  // ColorReconstruction.h:23
    if (s != cudaSuccess) return fail(e, VC_ERR_CUDA, "vc_set_images_raw: %s", cudaGetErrorString(s));
    return VC_OK;
}

int vc_append_views(vc_engine* e, int32_t n, const float* P, const float* M, const void* masks, int32_t mask_format, const uint8_t* images_bgr) {
    if (!e) return VC_ERR_ARG;
    // every check before any state changes
    if (e->V == 0 || !e->d_mask) return fail(e, VC_ERR_STATE, "vc_append_views: call vc_set_views and vc_set_masks first");
    if (mask_format != VC_MASK_BITS && mask_format != VC_MASK_BGR8 && mask_format != VC_MASK_BGR8_RAW) return fail(e, VC_ERR_ARG, "vc_append_views: unknown mask format %d", mask_format);
    if (mask_format == VC_MASK_BGR8_RAW && !e->have_calib) return fail(e, VC_ERR_STATE, "vc_append_views: raw masks need vc_set_calibration first");
    if (mask_format == VC_MASK_BGR8_RAW && (e->W > VC_RAW_MAX_SIDE || e->H > VC_RAW_MAX_SIDE))
        return fail(e, VC_ERR_ARG, "vc_append_views: raw masks of %dx%d: cv::undistort takes W and H up to %d", e->W, e->H, VC_RAW_MAX_SIDE);
    if (n < 1) return fail(e, VC_ERR_ARG, "vc_append_views: n=%d views (need at least 1)", n);
    if (!P || !masks) return fail(e, VC_ERR_ARG, "vc_append_views: P and masks are required");
    if ((long long)e->V + n > VC_MAX_TOTAL_VIEWS) return fail(e, VC_ERR_ARG, "vc_append_views: %d + %d views exceed %d", e->V, n, VC_MAX_TOTAL_VIEWS);
    const int V1 = e->V + n;
    const size_t view_words = (size_t)e->H * e->Ww, view_bgr = (size_t)e->H * e->W * 3;
    if ((size_t)V1 * view_words > 0x7fffffffull) return fail(e, VC_ERR_ARG, "vc_append_views: %d views of %dx%d exceed 2^31 mask words", V1, e->W, e->H);
    if ((M != nullptr) != e->have_M) return fail(e, VC_ERR_ARG, "vc_append_views: M must be given if and only if the engine's views have M (%s)", e->have_M ? "they do" : "they do not");
    if ((images_bgr != nullptr) != (e->d_images != nullptr))
        return fail(e, VC_ERR_ARG, "vc_append_views: images must be given if and only if the engine holds images (%s)", e->d_images ? "it does" : "it does not");
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaStreamSynchronize(e->stream));  // earlier work may still read the host view vectors and the buffers replaced below
    // host side of the new views
    std::vector<VcViewConst> hv(e->h_view);
    std::vector<float> hc(e->h_cam);
    std::vector<VcViewFilter> hf(e->h_filt);
    hv.resize(V1); hc.resize((size_t)V1 * 4, 0.0f); hf.resize(V1, VcViewFilter{});
    for (int i = 0; i < n; i++) {
        const int v = e->V + i;
        for (int k = 0; k < 12; k++) hv[v].P[k] = (double)P[i * 12 + k];
        for (int k = 0; k < 12; k++) hf[v].P[k] = P[i * 12 + k];
        if (M) { hc[v * 4 + 0] = M[i * 12 + 3]; hc[v * 4 + 1] = M[i * 12 + 7]; hc[v * 4 + 2] = M[i * 12 + 11]; hc[v * 4 + 3] = 1.0f; }
    }
    vc_filter_constants(e, hf.data() + e->V, n);  // (it also rewrites hDu / hDv, which depend on W and H only: same values)
    // new buffers for all V1 views; the engine's own are replaced only once everything has succeeded
    const bool raw = mask_format == VC_MASK_BGR8_RAW;
    const size_t sat_view = (size_t)(e->H + 1) * vc_sat_pitch(e->W);
    uint32_t *mask = nullptr, *sat_tmp = nullptr;
    vc_sat_t* sat = nullptr;
    uint8_t *images = nullptr, *stage = nullptr;
    VcViewFilter* filt = nullptr;
    VcViewConst* view64 = nullptr;
    float4* cam = nullptr;
    const size_t stage_bytes = mask_format != VC_MASK_BITS ? (size_t)n * view_bgr * (raw ? 2 : 1) : 0;  // 8UC3 masks [+ undistorted copy]; raw images reuse it
    cudaError_t s = cudaMalloc(&mask, (size_t)V1 * view_words * 4);
    if (s == cudaSuccess) s = cudaMalloc(&sat_tmp, (size_t)V1 * view_words * 4);
    if (s == cudaSuccess) s = cudaMalloc(&sat, (size_t)V1 * sat_view * sizeof(vc_sat_t));
    if (s == cudaSuccess && images_bgr) s = cudaMalloc(&images, (size_t)V1 * view_bgr);
    if (s == cudaSuccess && stage_bytes) s = cudaMalloc(&stage, stage_bytes);
    // never fewer than VC_MAX_VIEWS entries: a later vc_set_views writes up to that many into these buffers without reallocating
    const size_t view_cap = (size_t)std::max(V1, VC_MAX_VIEWS);
    if (s == cudaSuccess) s = cudaMalloc(&filt, view_cap * sizeof(VcViewFilter));
    if (s == cudaSuccess) s = cudaMalloc(&view64, view_cap * sizeof(VcViewConst));
    if (s == cudaSuccess) s = cudaMalloc(&cam, (size_t)V1 * sizeof(float4));
    // the earlier views' masks, tables and images as they are, the new views' after them
    if (s == cudaSuccess) s = cudaMemcpyAsync(mask, e->d_mask, e->mask_bytes, cudaMemcpyDeviceToDevice, e->stream);
    if (s == cudaSuccess) s = cudaMemcpyAsync(sat, e->d_sat, (size_t)e->V * sat_view * sizeof(vc_sat_t), cudaMemcpyDeviceToDevice, e->stream);
    if (s == cudaSuccess && images_bgr) s = cudaMemcpyAsync(images, e->d_images, (size_t)e->V * view_bgr, cudaMemcpyDeviceToDevice, e->stream);
    if (s == cudaSuccess) s = cudaMemcpyAsync(filt, hf.data(), (size_t)V1 * sizeof(VcViewFilter), cudaMemcpyHostToDevice, e->stream);
    if (s == cudaSuccess) s = cudaMemcpyAsync(view64, hv.data(), (size_t)V1 * sizeof(VcViewConst), cudaMemcpyHostToDevice, e->stream);
    if (s == cudaSuccess) s = cudaMemcpyAsync(cam, hc.data(), (size_t)V1 * sizeof(float4), cudaMemcpyHostToDevice, e->stream);
    const uint8_t* bgr = nullptr;  // the new views' 8UC3 masks on the device
    if (s == cudaSuccess) {
        if (mask_format == VC_MASK_BITS) {
            s = cudaMemcpyAsync(mask + (size_t)e->V * view_words, masks, (size_t)n * view_words * 4, cudaMemcpyDefault, e->stream);  // host or device memory
        } else {
            s = cudaMemcpyAsync(stage, masks, (size_t)n * view_bgr, cudaMemcpyHostToDevice, e->stream);
            bgr = stage;
            if (s == cudaSuccess && raw) {  // cv::undistort(mask, ...) (VoxelCarving.cpp:36)
                s = undistort_device(stage, stage + (size_t)n * view_bgr, n, e->W, e->H, e->calib_K, e->calib_dist, e->stream, &e->d_undist_ir, &e->undist_ir_count);
                bgr = stage + (size_t)n * view_bgr;
            }
        }
    }
    if (s == cudaSuccess) s = build_view_tables(e, bgr, mask, sat_tmp, sat, e->V, V1);
    if (s == cudaSuccess && images_bgr) {
        uint8_t* dst = images + (size_t)e->V * view_bgr;
        if (raw) {  // ColorReconstruction.h:23
            s = cudaMemcpyAsync(stage, images_bgr, (size_t)n * view_bgr, cudaMemcpyHostToDevice, e->stream);
            if (s == cudaSuccess) s = undistort_device(stage, dst, n, e->W, e->H, e->calib_K, e->calib_dist, e->stream, &e->d_undist_ir, &e->undist_ir_count);
        } else {
            s = cudaMemcpyAsync(dst, images_bgr, (size_t)n * view_bgr, cudaMemcpyHostToDevice, e->stream);
        }
    }
    if (s == cudaSuccess) s = cudaStreamSynchronize(e->stream);  // the host vectors above are locals, and any error surfaces here
    cudaFree(stage);
    if (s != cudaSuccess) {
        cudaGetLastError();
        cudaFree(mask); cudaFree(sat_tmp); cudaFree(sat); cudaFree(images); cudaFree(filt); cudaFree(view64); cudaFree(cam);
        return fail(e, VC_ERR_CUDA, "vc_append_views: %s (the engine is unchanged)", cudaGetErrorString(s));
    }
    cudaFree(e->d_mask); cudaFree(e->d_sat_tmp); cudaFree(e->d_sat); cudaFree(e->d_filt); cudaFree(e->d_view64); cudaFree(e->d_cam);
    e->d_mask = mask; e->d_sat_tmp = sat_tmp; e->d_sat = sat; e->d_filt = filt; e->d_view64 = view64; e->d_cam = cam;
    if (images_bgr) { cudaFree(e->d_images); e->d_images = images; }
    e->h_view.swap(hv); e->h_cam.swap(hc); e->h_filt.swap(hf);
    e->V = V1;
    e->mask_bytes = (size_t)V1 * view_words * 4;
    e->views_version++;
    return VC_OK;
}

int vc_download_masks(vc_engine* e, uint32_t* bits) {
    if (!e) return VC_ERR_ARG;
    if (!bits) return fail(e, VC_ERR_ARG, "vc_download_masks: null buffer");
    if (!e->d_mask) return fail(e, VC_ERR_STATE, "vc_download_masks: no masks set");
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaMemcpyAsync(bits, e->d_mask, e->mask_bytes, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

int vc_download_images(vc_engine* e, uint8_t* images_bgr) {
    if (!e) return VC_ERR_ARG;
    if (!images_bgr) return fail(e, VC_ERR_ARG, "vc_download_images: null buffer");
    if (!e->d_images) return fail(e, VC_ERR_STATE, "vc_download_images: no images set");
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaMemcpyAsync(images_bgr, e->d_images, (size_t)e->V * e->H * e->W * 3, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

int vc_undistort_bgr(int32_t device, int32_t n, int32_t W, int32_t H, const uint8_t* src, const double K[9], const double* dist, int32_t n_dist, uint8_t* dst) {
    if (!src || !dst || !K || !dist || n < 1 || W < 1 || H < 1) return fail(nullptr, VC_ERR_ARG, "vc_undistort_bgr: bad argument");
    if (n_dist != 4 && n_dist != 5 && n_dist != 8) return fail(nullptr, VC_ERR_ARG, "vc_undistort_bgr: %d distortion coefficients (need 4, 5 or 8)", n_dist);
    if (W > VC_RAW_MAX_SIDE || H > VC_RAW_MAX_SIDE) return fail(nullptr, VC_ERR_ARG, "vc_undistort_bgr: %dx%d: cv::undistort takes W and H up to %d", W, H, VC_RAW_MAX_SIDE);
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return fail(nullptr, VC_ERR_CUDA, "vc_undistort_bgr: no CUDA device %d; this engine has no CPU fallback", device); }
    double d8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < n_dist; i++) d8[i] = dist[i];
    const size_t bytes = (size_t)n * H * W * 3;
    uint8_t *d_src = nullptr, *d_dst = nullptr;
    cudaError_t s = cudaMalloc(&d_src, bytes);
    if (s == cudaSuccess) s = cudaMalloc(&d_dst, bytes);
    if (s == cudaSuccess) s = cudaMemcpy(d_src, src, bytes, cudaMemcpyHostToDevice);
    if (s == cudaSuccess) s = undistort_device(d_src, d_dst, n, W, H, K, d8, 0);
    if (s == cudaSuccess) s = cudaMemcpy(dst, d_dst, bytes, cudaMemcpyDeviceToHost);
    cudaFree(d_src); cudaFree(d_dst);
    if (s != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_undistort_bgr: %s", cudaGetErrorString(s));
    return VC_OK;
}

int vc_reset(vc_engine* e) {
    if (!e) return VC_ERR_ARG;
    e->reset_pending = true;  // lazy: vc_carve(VC_EXACT) folds it into its coalesced fill pass
    e->flags_valid = false;
    e->carved_implies_seen = true;
    e->gathered = false;
    e->halo_lo = e->halo_hi = false;
    e->have_colors = false;
    e->have_mc = false;
    return VC_OK;
}

// The brick grid of `nz` planes of the slab (bricks of VC_BX x VC_BY x VC_BZ voxels, VC_BX = 32: one brick per word column)
// and the super-brick grid over it (VC_SUPER^3 bricks each)
struct BrickGeom {
    int nbx, nby, nbz, sbx, sby, sbz;
    long long n_bricks, n_super;
};
static BrickGeom brick_geom(const vc_engine* e, int nz) {
    BrickGeom b;
    b.nbx = e->Wx; b.nby = (e->g.Y + VC_BY - 1) / VC_BY; b.nbz = (nz + VC_BZ - 1) / VC_BZ;
    b.sbx = (b.nbx + VC_SUPER - 1) / VC_SUPER; b.sby = (b.nby + VC_SUPER - 1) / VC_SUPER; b.sbz = (b.nbz + VC_SUPER - 1) / VC_SUPER;
    b.n_bricks = (long long)b.nbx * b.nby * b.nbz;
    b.n_super = (long long)b.sbx * b.sby * b.sbz;
    return b;
}

// Buffers of the brick classifier, sized for the whole slab (a z-chunk uses a prefix of each).
static int ensure_brick_buffers(vc_engine* e) {
    const BrickGeom b = brick_geom(e, e->nz);
    if (b.n_bricks > 0x7fffffffLL) return fail(e, VC_ERR_ARG, "slab too large for one launch (%lld bricks)", b.n_bricks);
    const long long n_super = (long long)b.sbx * b.sby * (b.sbz + 1);
    if (e->resident_blocks < 1) {  // persistent grid of vc_carve_bricks: as many blocks of 8 warps as are resident at once
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&e->resident_blocks, vc_carve_bricks<false>, 256, 0) != cudaSuccess || e->resident_blocks < 1) { cudaGetLastError(); e->resident_blocks = 2; }
    }
    if (!e->fill_stream) {
        VC_CUDA(e, cudaStreamCreateWithFlags(&e->fill_stream, cudaStreamNonBlocking));
        VC_CUDA(e, cudaEventCreateWithFlags(&e->ev_fill_fork, cudaEventDisableTiming));
        VC_CUDA(e, cudaEventCreateWithFlags(&e->ev_fill_join, cudaEventDisableTiming));
    }
    if (e->d_bricks) return VC_OK;
    VC_CUDA(e, cudaMalloc(&e->d_bricks, (size_t)b.n_bricks * sizeof(VcBrickState)));
    VC_CUDA(e, cudaMalloc(&e->d_super, (size_t)n_super * sizeof(VcBrickState)));
    VC_CUDA(e, cudaMalloc(&e->d_brick_flags, (size_t)b.n_bricks));
    VC_CUDA(e, cudaMalloc(&e->d_super_flags, (size_t)n_super));
    VC_CUDA(e, cudaMalloc(&e->d_super_list, (size_t)n_super * sizeof(unsigned int)));
    return VC_OK;
}

static VcCarveParams carve_params(vc_engine* e, int view_begin, int view_end) {
    const int K = 4;
    VcCarveParams p{};
    p.occ = e->occ_slab(); p.seen = e->seen_slab(); p.mask = e->d_mask;
    p.executed = e->d_scalars + 2;
    p.X = e->g.X; p.Y = e->g.Y; p.Wx = e->Wx; p.G = (e->Wx + K - 1) / K;
    p.YB = (e->g.Y + VC_TILE_ROWS - 1) / VC_TILE_ROWS;
    p.z_begin = e->g.z_begin; p.nz = e->nz;
    p.W = e->W; p.H = e->H; p.Ww = e->Ww;
    p.mask_plane = (uint32_t)((size_t)e->H * e->Ww);
    p.v0 = view_begin; p.v1 = view_end;
    p.s = e->g.voxel_size;
    p.hDu = e->hDu; p.hDv = e->hDv;
    return p;
}

// The part of the view range [v0, v1) that lies in view group g, as carve parameters relative to the group's first view: the
// kernels index the constant tables and the per-view buffers from there, so their view offsets stay what they are for one group.
static VcCarveParams group_params(const vc_engine* e, VcCarveParams p, int g, int v0, int v1) {
    const int base = g * VC_MAX_VIEWS;
    p.v0 = std::max(v0, base) - base;
    p.v1 = std::max(std::min(v1, base + VC_MAX_VIEWS) - base, p.v0);
    p.mask = e->d_mask + (size_t)base * p.mask_plane;
    return p;
}
// the view groups [g0, g1] that [v0, v1) intersects; an empty range still gets the group of v0 (a fresh carve writes the reset)
static void group_span(const vc_engine* e, int v0, int v1, int& g0, int& g1) {
    g0 = std::min(v0, e->V - 1) / VC_MAX_VIEWS;
    g1 = v1 > v0 ? (v1 - 1) / VC_MAX_VIEWS : g0;
}

// Both levels of the brick classifier on the planes [z_begin, z_begin + nz) of the grid (geometry b), for the views [v0, v1) of
// the group whose tables start at view vbase: the list lengths are reset, the super-bricks classified into the dense array,
// then the bricks of the undecided ones into the flags and the work list.  executed: the corner-projection counter of a
// counting run, or null.  pdl: level 0 may start while level 1 drains.
static int classify_bricks(vc_engine* e, const BrickGeom& b, int z_begin, int nz, int v0, int v1, int vbase, unsigned long long* executed, bool pdl) {
    unsigned int* d_nlist = (unsigned int*)(e->d_scalars + 6);  // [6] = front list length | super-list length, [7] = work counter | back list length
    VC_CUDA(e, cudaMemsetAsync(e->d_scalars + 6, 0, 2 * sizeof(unsigned long long), e->stream));
    VcBrickParams bp{};
    bp.list = e->d_bricks; bp.n_list = d_nlist; bp.n_list_back = d_nlist + 3; bp.list_cap = (unsigned)b.n_bricks;
    bp.brick_flags = e->d_brick_flags; bp.sat = e->d_sat + (size_t)vbase * (e->H + 1) * vc_sat_pitch(e->W);
    bp.super_flags = e->d_super_flags; bp.super_list = e->d_super_list; bp.n_super_list = d_nlist + 1;
    bp.executed = executed;
    bp.X = e->g.X; bp.Y = e->g.Y; bp.Wx = e->Wx; bp.nz = nz; bp.z_begin = z_begin;
    bp.nbx = b.nbx; bp.nby = b.nby; bp.nbz = b.nbz; bp.W = e->W; bp.H = e->H; bp.v0 = v0; bp.v1 = v1; bp.s = e->g.voxel_size;
    VcBrickParams sp = bp;  // level 1: super-bricks into the dense array
    sp.dense = e->d_super; sp.nbx = b.sbx; sp.nby = b.sby; sp.nbz = b.sbz;
    vc_brick_classify_kernel<1><<<(unsigned)((b.n_super + VC_CLS_L1_CH - 1) / VC_CLS_L1_CH), 256, 0, e->stream>>>(sp);  // VC_CLS_L1_CH super-bricks per block
    bp.dense = e->d_super; bp.pbx = b.sbx; bp.pby = b.sby;
    // level 0: the blocks walk the list of undecided super-bricks (length known on the device only)
    const long long l0_grid = std::min<long long>(b.n_super, 8LL * e->sm_count);
    VC_CUDA(e, launch_pdl(vc_brick_classify_kernel<0>, dim3((unsigned)l0_grid), dim3(VC_CLS_L0_THREADS), e->stream, pdl, bp));
    return VC_OK;
}

// VC_EXACT on the planes [zl0, zl1) of the slab (zl0 a multiple of the super-brick height, so bricks sit where they
// would in a whole-slab pass): classify super-bricks, classify bricks, fill, evaluate the undecided pairs.  vbase: first view
// of the group whose constants are loaded (p from group_params); the per-view device arrays are read from there.
static int carve_exact_range(vc_engine* e, VcCarveParams p, int zl0, int zl1, bool count, bool fresh, bool record_mid, int vbase = 0) {
    const long long off = (long long)zl0 * e->plane_words;
    p.occ += off; p.seen += off;
    p.z_begin = e->g.z_begin + zl0; p.nz = zl1 - zl0;
    const BrickGeom b = brick_geom(e, p.nz);
    if (p.nz > 65535) return fail(e, VC_ERR_ARG, "vc_carve: slab of %d planes exceeds the fill grid", p.nz);
    unsigned int* d_work = (unsigned int*)(e->d_scalars + 7);
    const bool quads = e->Wx % 4 == 0;
    const unsigned Q = (unsigned)e->Wx / 4u;  // quads per row
    int q_shift = -1;                         // log2(Q) when the rows are whole quads and Q is a power of two
    if (quads) for (int k = 0; k < 31; k++) if (Q == (1u << k)) q_shift = k;
    // Fresh carve: most words end up "carved and seen".  That pattern is written everywhere first, by a kernel that needs nothing
    // from the classification and runs next to it on a second stream (a fork / join the graph capture follows); the fill pass
    // inside vc_carve_bricks then only writes the words of bricks that are neither carved nor listed.
    bool fill_forked = false;
    if (fresh && quads) {
        const int rem = e->g.X - (e->Wx - 1) * 32;
        const size_t n_quads = (size_t)p.nz * e->g.Y * Q;
        // As a branch of the captured graph it runs next to the classification.  Plain launches (profiling mode, VOXCARVE_NO_GRAPH,
        // the z-chunks of vc_carve_download) keep it in stream order instead: queued up behind a running kernel, the two-stream
        // version of the same sequence measured up to 1.6x slower than the graph (tools/experiments/profile_split_probe.py), and
        // the two do not overlap anyway (both wait for the memory).
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        VC_CUDA(e, cudaStreamIsCapturing(e->stream, &cap));
        fill_forked = cap == cudaStreamCaptureStatusActive;
        cudaStream_t fs = fill_forked ? e->fill_stream : e->stream;
        if (fill_forked) {
            VC_CUDA(e, cudaEventRecord(e->ev_fill_fork, e->stream));
            VC_CUDA(e, cudaStreamWaitEvent(e->fill_stream, e->ev_fill_fork, 0));
        }
        const unsigned bgrid = (unsigned)std::min<size_t>((n_quads + 255) / 256, (size_t)e->sm_count);  // one block per SM reaches the memory's write rate and leaves room for the classification's blocks
        vc_blind_fill_kernel<<<bgrid, 256, 0, fs>>>((uint4*)p.occ, (uint4*)p.seen, n_quads, Q, q_shift, rem >= 32 ? 0xffffffffu : ((1u << rem) - 1u));
        VC_CUDA(e, cudaGetLastError());
        if (fill_forked) VC_CUDA(e, cudaEventRecord(e->ev_fill_join, e->fill_stream));
    }
    // level 0 overlaps level 1 unless the mid-point event is recorded: an event record would keep the kernels apart anyway
    int rc =classify_bricks(e, b, p.z_begin, p.nz, p.v0, p.v1, vbase, count ? e->d_scalars + 5 : nullptr, !record_mid);
    if (rc) return rc;
    if (record_mid) VC_CUDA(e, cudaEventRecord(e->evm, e->stream));  // (profiling / counting runs only: it sits between two kernels that otherwise overlap their launch)
    const unsigned pgrid = (unsigned)e->sm_count * (unsigned)e->resident_blocks;  // persistent grid (ensure_brick_buffers)
    // Fill pass (volume words implied by the brick flags).  Fresh carve, rows of whole quads: the first blocks of the persistent
    // kernel patch what the blind fill got wrong, skipping the listed bricks, whose words the work items own.  Otherwise it runs
    // first, in stream order (it must apply the flags before the per-voxel kernel reads the state; rows of other widths go word
    // by word).
    VcFillParams fp{};
    fp.occ = p.occ; fp.seen = p.seen; fp.brick_flags = e->d_brick_flags; fp.super_flags = e->d_super_flags;
    fp.X = e->g.X; fp.Y = e->g.Y; fp.Wx = e->Wx; fp.nby = b.nby; fp.pbx = b.sbx; fp.pby = b.sby;
    fp.nz = p.nz; fp.q_shift = q_shift; fp.n_fill_blocks = 0;
    if (fill_forked) VC_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_fill_join, 0));  // before anything else writes the volumes
    if (quads) fp.per_plane = (unsigned)(((long long)e->g.Y * Q + 255) / 256);
    if (fresh && quads) {
        // ONE fill block per SM (blocks are dealt round-robin).  More of them when the slab has many brick layers was the r1
        // heuristic; measured on C5 (256 layers): 1 / 2 / 3 / 4 fill blocks per SM = 1.90 / 1.96 / 1.99 / 2.02 ms - the kernel is
        // bound by its computing blocks, so the fill gets as few as keep the stores flowing.
        fp.n_fill_blocks = std::min((unsigned)e->sm_count, pgrid);
    } else if (quads) {
        vc_fill4_kernel<<<dim3(fp.per_plane, (unsigned)b.nbz), 256, 0, e->stream>>>(fp);  // one block per (256 quads, brick layer)
    } else {
        vc_fill_kernel<<<dim3((e->g.Y + 7) / 8, p.nz, (e->Wx + 31) / 32), dim3(32, 8), 0, e->stream>>>(
            p.occ, p.seen, e->d_brick_flags, e->d_super_flags, e->g.X, e->g.Y, e->Wx, b.nby, b.sbx, b.sby, fresh ? 1 : 0, 0);
    }
    // The per-voxel kernel is launched plainly, onto an empty GPU.  Its fill pass relies on the first blocks of the grid landing
    // on different SMs (one fill block per SM, HBM-bound, next to three computing blocks); as a programmatic dependent launch
    // its blocks take whatever slots the classification frees first, the fill blocks pile up on a few SMs, and slabs that are
    // mostly fill get 30 % slower (C5, slab 0 of 8: 0.30 -> 0.39 ms).  Only the level-0 classification overlaps its predecessor.
    const unsigned int* d_nlist = (const unsigned int*)(e->d_scalars + 6);
    const vc_sat_t* sat = e->d_sat + (size_t)vbase * (e->H + 1) * vc_sat_pitch(e->W);
    if (count) vc_carve_bricks<true><<<pgrid, 256, 0, e->stream>>>(p, e->d_bricks, d_nlist, d_work + 1, (unsigned)b.n_bricks, d_work, b.nbx, b.nby, sat, fresh ? 1 : 0, e->d_filt + vbase, e->d_view64 + vbase, fp);
    else vc_carve_bricks<false><<<pgrid, 256, 0, e->stream>>>(p, e->d_bricks, d_nlist, d_work + 1, (unsigned)b.n_bricks, d_work, b.nbx, b.nby, sat, fresh ? 1 : 0, e->d_filt + vbase, e->d_view64 + vbase, fp);
    VC_CUDA(e, cudaGetLastError());
    e->stats.carve_launches += 4;  // blind fill or fill pass, two classification levels, per-voxel kernel
    return VC_OK;
}

// One carve of the views [v0, v1) on the planes [zl0, zl1) of the slab, view group by view group: each group's constants are
// uploaded in stream order behind the previous group's kernels, and only the first group starts from a pending reset (`fresh`);
// the others accumulate onto its result.  With one group (at most VC_MAX_VIEWS views) this is one plain sequence.  Counting
// runs of VC_EXACT add the bricks each group listed for per-voxel work to *listed.
static int carve_groups(vc_engine* e, int32_t mode, const VcCarveParams& p, int v0, int v1, int zl0, int zl1, bool count, bool fresh,
                        bool record_mid, uint64_t* listed) {
    int g0, g1;
    group_span(e, v0, v1, g0, g1);
    for (int g = g0; g <= g1; g++) {
        int rc = ensure_constants(e, g);
        if (rc) return rc;
        const VcCarveParams pg = group_params(e, p, g, v0, v1);
        if (mode == VC_EXACT) rc = carve_exact_range(e, pg, zl0, zl1, count, fresh && g == g0, record_mid, g * VC_MAX_VIEWS);
        else rc = launch_carve<4>(e, mode == VC_EXACT_FLAT ? VC_EXACT : mode, pg, count);
        if (rc) return rc;
        if (count && mode == VC_EXACT) {  // the next group resets the list lengths
            unsigned long long nl = 0, nw = 0;
            VC_CUDA(e, cudaMemcpyAsync(&nl, e->d_scalars + 6, sizeof nl, cudaMemcpyDeviceToHost, e->stream));
            VC_CUDA(e, cudaMemcpyAsync(&nw, e->d_scalars + 7, sizeof nw, cudaMemcpyDeviceToHost, e->stream));
            VC_CUDA(e, cudaStreamSynchronize(e->stream));
            *listed += (nl & 0xffffffffull) + (nw >> 32);  // front + back of the work list
        }
    }
    return VC_OK;
}

// after the last kernel of a carve (vc_carve, vc_carve_download): its end event, the view constants released, the per-call
// statistics reset, and everything derived from the volumes marked stale
static int carve_finish(vc_engine* e, uint64_t nominal_voxel_views) {
    VC_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    int rc = constants_used(e);
    if (rc) return rc;
    e->stats.nominal_voxel_views = nominal_voxel_views;
    e->stats.executed_voxel_views = 0;
    e->stats.brick_corner_views = 0;
    e->stats.filter_rows = e->stats.filter_slow_rows = e->stats.filter_mismatches = e->stats.subbrick_corner_views = 0;
    e->stats.last_carve_ms = -1.0;  // resolved lazily in vc_get_stats
    e->gathered = false;
    e->halo_lo = e->halo_hi = false;  // the neighbours carve too: their planes are stale
    e->have_colors = false;
    e->have_mc = false;
    return VC_OK;
}

static int carve_check(vc_engine* e, const char* who, int32_t mode, int32_t& view_begin, int32_t& view_end) {
    if (mode != VC_EXACT && mode != VC_FAST_F32 && mode != VC_EXACT_FLAT) return fail(e, VC_ERR_ARG, "%s: unknown mode %d", who, mode);
    if (e->V == 0 || !e->d_mask) return fail(e, VC_ERR_STATE, "%s: views and masks must be set first", who);
    if (view_end < 0) view_end = e->V;
    if (view_begin < 0 || view_begin > view_end || view_end > e->V)
        return fail(e, VC_ERR_ARG, "%s: bad view range [%d,%d) for V=%d", who, view_begin, view_end, e->V);
    if (bind_device(e)) return VC_ERR_CUDA;
    int rc = ensure_volumes(e);
    if (rc) return rc;
    return e->V > VC_MAX_VIEWS ? VC_OK : ensure_constants(e);  // several groups: uploaded group by group
}

// NVTX range named after a phase of the reference's Benchmark singleton (Benchmark.h:86-124): Carving, Coloring,
// PostProcessing, MarchingCubes - what a profiler timeline of a -c=5 / -c=6 run shows next to the reference's own phases
struct PhaseRange {
    explicit PhaseRange(const char* name) { nvtxRangePushA(name); }
    ~PhaseRange() { nvtxRangePop(); }
};

int vc_carve(vc_engine* e, int32_t mode, int32_t view_begin, int32_t view_end, int32_t count_executed) {
    if (!e) return VC_ERR_ARG;
    PhaseRange nvtx("Carving");
    int rc = carve_check(e, "vc_carve", mode, view_begin, view_end);
    if (rc) return rc;
    VcCarveParams p = carve_params(e, view_begin, view_end);
    if (count_executed) VC_CUDA(e, cudaMemsetAsync(e->d_scalars + 2, 0, sizeof(unsigned long long), e->stream));
    if (count_executed) VC_CUDA(e, cudaMemsetAsync(e->d_scalars + 5, 0, sizeof(unsigned long long), e->stream));
    if (count_executed) VC_CUDA(e, cudaMemsetAsync(e->d_scalars + 8, 0, 4 * sizeof(unsigned long long), e->stream));
    if (mode == VC_EXACT) { rc = ensure_brick_buffers(e); if (rc) return rc; }
    if (mode != VC_EXACT) { rc = materialize_reset(e); if (rc) return rc; }
    // Every kernel skips voxels that are already carved, which is exact as long as carved => seen.  An uploaded state may hold
    // voxels that are carved but unseen; the reference still projects those and marks them seen (VoxelCarving.cpp:45-54).  They
    // are carved as if occupied (so their `seen` bit comes out right; a carved voxel is seen by the view that carved it) and
    // the uploaded occupancy is and-ed back afterwards.
    uint32_t* d_saved_occ = nullptr;
    if (!e->carved_implies_seen && !e->reset_pending) {
        void* sc = nullptr;
        rc = ensure_scratch(e, (size_t)e->slab_words * 4, &sc);
        if (rc) return rc;
        d_saved_occ = (uint32_t*)sc;
        vc_unseen_begin_kernel<<<(unsigned)((e->slab_words + 255) / 256), 256, 0, e->stream>>>(e->occ_slab(), e->seen_slab(), d_saved_occ, e->slab_words, e->Wx, e->g.X);
        VC_CUDA(e, cudaGetLastError());
    }
    VC_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    e->stats.bricks_total = mode == VC_EXACT ? (uint64_t)brick_geom(e, e->nz).n_bricks : 0;
    e->stats.bricks_listed = 0;
    uint64_t listed = 0;  // counting run of VC_EXACT: listed bricks summed over the view groups
    const bool fresh = mode == VC_EXACT && e->reset_pending;
    if (mode == VC_EXACT && e->use_graphs < 0) { const char* ng = getenv("VOXCARVE_NO_GRAPH"); e->use_graphs = (ng && atoi(ng) != 0) ? 0 : 1; }
    // a whole-range VC_EXACT carve of one view group (its constants uploaded by carve_check) is one cached CUDA graph
    const bool graph = mode == VC_EXACT && e->use_graphs && !e->profiling && !count_executed && view_begin == 0 && view_end == e->V &&
                       e->V <= VC_MAX_VIEWS;
    e->have_mid = mode == VC_EXACT && !graph && e->V <= VC_MAX_VIEWS && (e->profiling || count_executed != 0);
    if (graph) {
        CarveGraphKey k;
        memset(&k, 0, sizeof k);  // padding bytes too: the key is compared with memcmp
        k.p = p;
        const void* ptrs[10] = {e->d_bricks, e->d_super, e->d_brick_flags, e->d_super_flags, e->d_super_list, e->d_sat, e->d_filt, e->d_view64, e->d_scalars, e->evm};
        memcpy(k.ptrs, ptrs, sizeof ptrs);
        k.fresh = fresh ? 1 : 0; k.sm_count = e->sm_count;
        CarveGraphSlot& gs = e->graph_slot[fresh ? 1 : 0];
        bool captured_now = false;
        if (!gs.valid || memcmp(&gs.key, &k, sizeof k) != 0) {
            captured_now = true;
            if (gs.exec) { cudaGraphExecDestroy(gs.exec); gs.exec = nullptr; }
            gs.valid = false;
            cudaGraph_t g = nullptr;
            VC_CUDA(e, cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
            rc = carve_exact_range(e, p, 0, e->nz, false, fresh, false);
            const cudaError_t ce = cudaStreamEndCapture(e->stream, &g);  // always end the capture, also after a failed launch
            if (rc) { if (g) cudaGraphDestroy(g); return rc; }
            if (ce != cudaSuccess) return fail(e, VC_ERR_CUDA, "vc_carve: stream capture failed: %s", cudaGetErrorString(ce));
            const cudaError_t ci = cudaGraphInstantiate(&gs.exec, g, 0);
            cudaGraphDestroy(g);
            if (ci != cudaSuccess) { gs.exec = nullptr; return fail(e, VC_ERR_CUDA, "vc_carve: cudaGraphInstantiate failed: %s", cudaGetErrorString(ci)); }
            gs.key = k;
            gs.valid = true;
        }
        VC_CUDA(e, cudaGraphLaunch(gs.exec, e->stream));
        if (!captured_now) e->stats.carve_launches += 4;  // the capture counted its own
    } else {
        rc = carve_groups(e, mode, p, view_begin, view_end, 0, e->nz, count_executed != 0, fresh, e->have_mid, &listed);
        if (rc) return rc;
    }
    if (mode == VC_EXACT) e->reset_pending = false;
    // the flags of a fresh whole-range VC_EXACT carve say everything about the volumes (with several groups, no single group's flags do)
    e->flags_valid = fresh && view_begin == 0 && view_end == e->V && e->V <= VC_MAX_VIEWS;
    if (d_saved_occ) {
        vc_unseen_end_kernel<<<(unsigned)((e->slab_words + 255) / 256), 256, 0, e->stream>>>(e->occ_slab(), d_saved_occ, e->slab_words);
        VC_CUDA(e, cudaGetLastError());
    }
    rc = carve_finish(e, (uint64_t)e->g.X * e->g.Y * e->nz * (uint64_t)(view_end - view_begin));
    if (rc) return rc;
    if (count_executed) {
        unsigned long long ex = 0, bc = 0, fl[4] = {0, 0, 0, 0};
        VC_CUDA(e, cudaMemcpyAsync(fl, e->d_scalars + 8, sizeof fl, cudaMemcpyDeviceToHost, e->stream));
        VC_CUDA(e, cudaMemcpyAsync(&ex, e->d_scalars + 2, sizeof ex, cudaMemcpyDeviceToHost, e->stream));
        VC_CUDA(e, cudaMemcpyAsync(&bc, e->d_scalars + 5, sizeof bc, cudaMemcpyDeviceToHost, e->stream));
        VC_CUDA(e, cudaStreamSynchronize(e->stream));
        e->stats.bricks_listed = listed;
        e->stats.executed_voxel_views = ex + (mode == VC_EXACT ? bc : 0);
        e->stats.brick_corner_views = mode == VC_EXACT ? bc : 0;
        if (mode == VC_EXACT) { e->stats.filter_rows = fl[0]; e->stats.filter_slow_rows = fl[1]; e->stats.filter_mismatches = fl[2]; e->stats.subbrick_corner_views = fl[3]; }
    }
    return VC_OK;
}

int vc_carve_download(vc_engine* e, int32_t mode, uint32_t* occupied, uint32_t* seen, uint64_t n_words) {
    if (!e) return VC_ERR_ARG;
    if (!occupied || !seen) return fail(e, VC_ERR_ARG, "vc_carve_download: null buffer");
    PhaseRange nvtx("Carving");
    if (n_words < (uint64_t)e->slab_words) return fail(e, VC_ERR_CAPACITY, "vc_carve_download: buffers hold %llu words, slab has %lld", (unsigned long long)n_words, e->slab_words);
    int32_t v0 = 0, v1 = -1;
    int rc = carve_check(e, "vc_carve_download", mode, v0, v1);
    if (rc) return rc;
    const int LZ = VC_BZ * VC_SUPER;
    int n_chunks = e->nz >= 8 * LZ ? 4 : (e->nz >= 2 * LZ ? 2 : 1);
    if (mode != VC_EXACT) n_chunks = 1;
    // a cudaMemcpyAsync into pageable memory blocks the host until the chunk has arrived, so the next chunk's kernels would
    // not be enqueued meanwhile: the chunked path only pays off with page-locked buffers (cudaHostAlloc / cudaHostRegister)
    if (!host_pinned(occupied) || !host_pinned(seen)) n_chunks = 1;
    if (!e->carved_implies_seen && !e->reset_pending) n_chunks = 1;  // uploaded state with carved-but-unseen voxels: vc_carve handles it
    if (n_chunks == 1) {  // nothing to overlap: plain sequence
        rc = vc_carve(e, mode, 0, -1, 0);
        if (!rc) rc = vc_download_occupied(e, occupied, n_words);
        if (!rc) rc = vc_download_seen(e, seen, n_words);
        return rc;
    }
    rc = ensure_brick_buffers(e);
    if (rc) return rc;
    if (!e->copy_stream) {
        VC_CUDA(e, cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        for (int c = 0; c < 4; c++) VC_CUDA(e, cudaEventCreateWithFlags(&e->ev_chunk[c], cudaEventDisableTiming));
    }
    VcCarveParams p = carve_params(e, v0, v1);
    const int cz = ((e->nz + n_chunks - 1) / n_chunks + LZ - 1) / LZ * LZ;  // planes per chunk, a multiple of the super-brick height
    VC_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    e->have_mid = false;
    e->stats.bricks_total = (uint64_t)brick_geom(e, e->nz).n_bricks;
    e->stats.bricks_listed = 0;
    const bool fresh = e->reset_pending;
    int c = 0;
    for (int zl0 = 0; zl0 < e->nz; zl0 += cz, c++) {
        const int zl1 = zl0 + cz < e->nz ? zl0 + cz : e->nz;
        rc = carve_groups(e, VC_EXACT, p, v0, v1, zl0, zl1, false, fresh, false, nullptr);  // the chunk's first group starts from the pending reset
        if (rc) return rc;
        VC_CUDA(e, cudaEventRecord(e->ev_chunk[c], e->stream));
        VC_CUDA(e, cudaStreamWaitEvent(e->copy_stream, e->ev_chunk[c], 0));
        const long long off = (long long)zl0 * e->plane_words, n = (long long)(zl1 - zl0) * e->plane_words;
        VC_CUDA(e, cudaMemcpyAsync(occupied + off, e->occ_slab() + off, n * 4, cudaMemcpyDeviceToHost, e->copy_stream));
        VC_CUDA(e, cudaMemcpyAsync(seen + off, e->seen_slab() + off, n * 4, cudaMemcpyDeviceToHost, e->copy_stream));
    }
    e->reset_pending = false;
    e->flags_valid = false;  // the flag arrays were re-used chunk by chunk
    rc = carve_finish(e, (uint64_t)e->g.X * e->g.Y * e->nz * (uint64_t)e->V);
    if (rc) return rc;
    VC_CUDA(e, cudaStreamSynchronize(e->copy_stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

// Sparse form of a FRESH carve: most bricks (C4: 96 %) are uniform - carved whole, or untouched - and are fully described by
// their flag byte; only the listed bricks (the ones vc_carve_bricks evaluated per voxel) need their words.  C4: 0.5 MB of
// flags + 10 MB of words instead of 268 MB over PCIe.
int vc_sparse_dims(const vc_engine* e, uint32_t* nbx, uint32_t* nby, uint32_t* nbz) {
    if (!e || !nbx || !nby || !nbz) return VC_ERR_ARG;
    const BrickGeom b = brick_geom(e, e->nz);
    *nbx = (uint32_t)b.nbx; *nby = (uint32_t)b.nby; *nbz = (uint32_t)b.nbz;
    return VC_OK;
}

int vc_carve_download_sparse(vc_engine* e, uint8_t* brick_flags, uint64_t flags_capacity, uint32_t* listed, uint32_t* words,
                             uint64_t listed_capacity, uint64_t* n_listed) {
    if (!e) return VC_ERR_ARG;
    PhaseRange nvtx("Carving");
    if (!brick_flags || !listed || !words || !n_listed) return fail(e, VC_ERR_ARG, "vc_carve_download_sparse: null argument");
    *n_listed = 0;
    const BrickGeom b = brick_geom(e, e->nz);
    const long long n_bricks = b.n_bricks;
    if (flags_capacity < (uint64_t)n_bricks) return fail(e, VC_ERR_CAPACITY, "vc_carve_download_sparse: flag buffer holds %llu bytes, the slab has %lld bricks", (unsigned long long)flags_capacity, n_bricks);
    if (!e->reset_pending) return fail(e, VC_ERR_STATE, "vc_carve_download_sparse: describes a carve that starts from the Model constructor state: call vc_reset first");
    int rc = vc_carve(e, VC_EXACT, 0, -1, 0);
    if (rc) return rc;
    void* sc = nullptr;
    rc = ensure_scratch(e, (size_t)n_bricks, &sc);  // resolved flags (the per-brick array is only written under undecided super-bricks)
    if (rc) return rc;
    uint8_t* d_flags = (uint8_t*)sc;
    if (e->V <= VC_MAX_VIEWS) {
        vc_sparse_flags_kernel<<<(unsigned)((n_bricks + 255) / 256), 256, 0, e->stream>>>(e->d_brick_flags, e->d_super_flags, d_flags, b.nbx, b.nby, b.nbz, b.sbx, b.sby);
    } else {  // several view groups: the flags and the list come from the volumes (the work list's front, its back left empty)
        VC_CUDA(e, cudaMemsetAsync(e->d_scalars + 6, 0, 2 * sizeof(unsigned long long), e->stream));
        vc_sparse_volume_flags_kernel<<<(unsigned)((n_bricks * 32 + 255) / 256), 256, 0, e->stream>>>(
            e->occ_slab(), e->seen_slab(), d_flags, e->d_bricks, (unsigned int*)(e->d_scalars + 6), e->g.X, e->g.Y, e->nz, e->Wx, b.nbx, b.nby, b.nbz);
    }
    VC_CUDA(e, cudaGetLastError());
    unsigned int counts[4] = {0, 0, 0, 0};  // front length, super-list length, work counter, back length
    VC_CUDA(e, cudaMemcpyAsync(counts, e->d_scalars + 6, sizeof counts, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaMemcpyAsync(brick_flags, d_flags, (size_t)n_bricks, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    const unsigned long long n = (unsigned long long)counts[0] + counts[3];
    *n_listed = n;
    if (n > listed_capacity) return fail(e, VC_ERR_CAPACITY, "vc_carve_download_sparse: %llu listed bricks, buffers hold %llu (volumes are complete on the device: vc_download_*)", n, (unsigned long long)listed_capacity);
    if (n == 0) return VC_OK;
    if (e->sparse_cap < n) {
        cudaFree(e->d_sparse_idx); cudaFree(e->d_sparse_words); e->d_sparse_idx = nullptr; e->d_sparse_words = nullptr; e->sparse_cap = 0;
        VC_CUDA(e, cudaMalloc(&e->d_sparse_idx, n * sizeof(uint32_t)));
        VC_CUDA(e, cudaMalloc(&e->d_sparse_words, n * 128 * sizeof(uint32_t)));
        e->sparse_cap = n;
    }
    vc_sparse_pack_kernel<<<(unsigned)((n + 3) / 4), 256, 0, e->stream>>>(e->d_bricks, counts[0], (unsigned)n, (unsigned)n_bricks, e->occ_slab(), e->seen_slab(),
                                                                         e->g.Y, e->nz, e->Wx, b.nbx, b.nby, e->d_sparse_idx, e->d_sparse_words);
    VC_CUDA(e, cudaGetLastError());
    VC_CUDA(e, cudaMemcpyAsync(listed, e->d_sparse_idx, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaMemcpyAsync(words, e->d_sparse_words, n * 128 * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

int vc_fast_carve(vc_engine* e, int32_t mode) {
    if (!e) return VC_ERR_ARG;
    PhaseRange nvtx("Carving");
    if (!e->whole_grid()) return fail(e, VC_ERR_STATE, "vc_fast_carve: the flood from voxel (0,0,0) needs the whole grid on one engine (slab [%d,%d) of Z=%d)", e->g.z_begin, e->g.z_end, e->g.Z);
    // refusals before the reset below: a refused call leaves the volumes as they were
    if (mode != VC_EXACT && mode != VC_FAST_F32 && mode != VC_EXACT_FLAT) return fail(e, VC_ERR_ARG, "vc_fast_carve: unknown mode %d", mode);
    if (e->V == 0 || !e->d_mask) return fail(e, VC_ERR_STATE, "vc_fast_carve: views and masks must be set first");
    // the set carve() would carve, on a fresh Model (fastCarve starts from the constructor state, main.cpp:248-264)
    int rc = vc_reset(e);
    if (rc) return rc;
    rc = vc_carve(e, mode, 0, -1, 0);
    if (rc) return rc;
    const long long n = e->slab_words;
    void* sc = nullptr;
    rc = ensure_scratch(e, (size_t)n * 4 + 16, &sc);
    if (rc) return rc;
    uint32_t* F = (uint32_t*)sc;
    int* d_changed = (int*)(F + n);
    VC_CUDA(e, cudaMemsetAsync(F, 0, n * 4 + 16, e->stream));
    uint32_t *occ = e->occ_slab(), *seen = e->seen_slab();
    const int X = e->g.X, Y = e->g.Y, Z = e->g.Z, Wx = e->Wx;
    vc_flood_seed_kernel<<<1, 1, 0, e->stream>>>(occ, F);
    const long long n_rows = (long long)Y * Z;
    // a round = sweeps along x, y, z; the device-side "changed" flag is read back only every VC_FLOOD_POLL rounds (a round after
    // convergence changes nothing, so at most VC_FLOOD_POLL - 1 rounds are wasted against a host round trip saved per round)
    const int VC_FLOOD_POLL = 4;
    int rounds = 0;
    for (;;) {
        if (rounds > 100000) return fail(e, VC_ERR_STATE, "vc_fast_carve: flood did not converge");
        VC_CUDA(e, cudaMemsetAsync(d_changed, 0, sizeof(int), e->stream));
        for (int k = 0; k < VC_FLOOD_POLL; k++, rounds++) {
            vc_flood_x_kernel<<<(unsigned)((n_rows + 127) / 128), 128, 0, e->stream>>>(occ, F, Wx, n_rows, X, d_changed);
            // along y: one thread per (z, word column); along z: one thread per (y, word column)
            vc_flood_axis_kernel<<<(unsigned)(((long long)Z * Wx + 127) / 128), 128, 0, e->stream>>>(occ, F, Wx, X, Y, Wx, (long long)Y * Wx, Z, d_changed);
            vc_flood_axis_kernel<<<(unsigned)(((long long)Y * Wx + 127) / 128), 128, 0, e->stream>>>(occ, F, Wx, X, Z, (long long)Y * Wx, Wx, Y, d_changed);
        }
        int h = 0;
        VC_CUDA(e, cudaMemcpyAsync(&h, d_changed, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
        VC_CUDA(e, cudaStreamSynchronize(e->stream));
        if (!h) break;
    }
    e->flags_valid = false;  // the flood rewrites the volumes
    vc_flood_finish_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(F, occ, seen, X, Y, Z, Wx);
    VC_CUDA(e, cudaGetLastError());
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stats.flood_rounds = (uint64_t)rounds;
    return VC_OK;
}

int vc_set_slab(vc_engine* e, int32_t z_begin, int32_t z_end) {
    if (!e) return VC_ERR_ARG;
    if (z_begin < 0 || z_end > e->g.Z || z_begin >= z_end) return fail(e, VC_ERR_ARG, "vc_set_slab: bad z-slab [%d,%d) for Z=%d", z_begin, z_end, e->g.Z);
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    e->g.z_begin = z_begin; e->g.z_end = z_end;
    e->nz = z_end - z_begin;
    e->slab_words = e->plane_words * e->nz;
    // everything sized by the slab is dropped and re-created on demand; views, masks and SAT stay
    vol_free(e->d_occ_own); vol_free(e->d_seen_own); e->d_occ_own = e->d_seen_own = nullptr;
    cudaFree(e->d_bricks); cudaFree(e->d_super); cudaFree(e->d_brick_flags); cudaFree(e->d_super_flags); cudaFree(e->d_super_list);
    e->d_bricks = nullptr; e->d_super = nullptr; e->d_brick_flags = nullptr; e->d_super_flags = nullptr; e->d_super_list = nullptr;
    cudaFree(e->d_block_sums);
    e->d_block_sums = nullptr;
    free_color(e);
    return vc_reset(e);
}

int vc_plan_slabs(vc_engine* e, int32_t n_parts, int32_t* z_bounds) {
    if (!e || !z_bounds) return VC_ERR_ARG;
    if (n_parts < 1 || n_parts > e->nz) return fail(e, VC_ERR_ARG, "vc_plan_slabs: n_parts=%d outside [1,%d]", n_parts, e->nz);
    if (e->V == 0 || !e->d_mask) return fail(e, VC_ERR_STATE, "vc_plan_slabs: views and masks must be set first");
    if (bind_device(e)) return VC_ERR_CUDA;
    int rc = VC_OK;
    for (int k = 0; k <= n_parts; k++) z_bounds[k] = e->g.z_begin + (int)((long long)k * e->nz / n_parts);  // uniform fallback
    const BrickGeom b = brick_geom(e, e->nz);
    const int nbz = b.nbz;
    if (nbz < n_parts) return VC_OK;  // fewer brick layers than parts: keep the uniform split
    rc = ensure_brick_buffers(e);
    if (rc) return rc;
    e->flags_valid = false;
    // both classification levels of VC_EXACT over the whole range, no volumes touched; once per view group, costs summed
    // cost of a brick layer (8 planes): per-voxel work of its listed bricks (undecided views x voxels) plus a small constant
    // per plane for the classification and fill passes
    std::vector<double> cost((size_t)nbz, 0.0);
    for (int grp = 0; grp < n_groups(e); grp++) {
        rc = ensure_constants(e, grp);
        if (rc) return rc;
        const int vbase = grp * VC_MAX_VIEWS;
        rc = classify_bricks(e, b, e->g.z_begin, e->nz, 0, std::min(VC_MAX_VIEWS, e->V - vbase), vbase, nullptr, false);
        if (rc) return rc;
        unsigned int counts[4] = {0, 0, 0, 0};  // front length, super-list length, (work counter), back length
        VC_CUDA(e, cudaMemcpyAsync(counts, e->d_scalars + 6, sizeof counts, cudaMemcpyDeviceToHost, e->stream));
        VC_CUDA(e, cudaStreamSynchronize(e->stream));
        std::vector<VcBrickState> h((size_t)counts[0] + counts[3]);  // the list is filled from both ends (VcBrickParams)
        if (counts[0]) VC_CUDA(e, cudaMemcpy(h.data(), e->d_bricks, (size_t)counts[0] * sizeof(VcBrickState), cudaMemcpyDeviceToHost));
        if (counts[3]) VC_CUDA(e, cudaMemcpy(h.data() + counts[0], e->d_bricks + (b.n_bricks - counts[3]), (size_t)counts[3] * sizeof(VcBrickState), cudaMemcpyDeviceToHost));
        for (const VcBrickState& st : h) cost[st.brick / ((unsigned)b.nbx * (unsigned)b.nby)] += (double)st.n_und * (VC_BX * VC_BY * VC_BZ);
    }
    // (every group's kernels are complete: its list was read back above)
    double total = 0.0;
    for (int z = 0; z < nbz; z++) total += cost[z];
    const double floor_cost = total > 0 ? 0.03 * total / nbz : 1.0;
    total = 0.0;
    for (int z = 0; z < nbz; z++) { cost[z] += floor_cost; total += cost[z]; }
    int layer = 0;
    double acc = 0.0;
    for (int k = 1; k < n_parts; k++) {
        const double target = total * k / n_parts;
        while (layer < nbz - (n_parts - k) && acc + cost[layer] * 0.5 < target) acc += cost[layer++];
        if (layer < k) { acc += cost[layer]; layer = k; }  // every part gets at least one layer
        z_bounds[k] = e->g.z_begin + layer * VC_BZ;
    }
    return VC_OK;
}

int vc_bind_volumes(vc_engine* e, void* d_occupied_full, void* d_seen_full) {
    if (!e) return VC_ERR_ARG;
    if (!d_occupied_full != !d_seen_full) return fail(e, VC_ERR_ARG, "vc_bind_volumes: bind both volumes or neither");
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    if (e->d_occ_full_own && d_occupied_full != e->d_occ_full_own) {  // replaces engine-owned whole-grid buffers
        vol_free(e->d_occ_full_own); vol_free(e->d_seen_full_own);
        e->d_occ_full_own = e->d_seen_full_own = nullptr;
    }
    e->d_occ_full = (uint32_t*)d_occupied_full;
    e->d_seen_full = (uint32_t*)d_seen_full;
    e->gathered = false;
    return vc_reset(e);
}

int vc_device_volumes(vc_engine* e, void** d_occupied_slab, void** d_seen_slab) {
    if (!e || !d_occupied_slab || !d_seen_slab) return VC_ERR_ARG;
    if (materialize_reset(e)) return VC_ERR_CUDA;
    *d_occupied_slab = e->occ_slab();
    *d_seen_slab = e->seen_slab();
    return VC_OK;
}

int vc_set_gathered(vc_engine* e, int32_t gathered) {
    if (!e) return VC_ERR_ARG;
    if (materialize_reset(e)) return VC_ERR_CUDA;
    if (gathered && !e->d_occ_full) return fail(e, VC_ERR_STATE, "vc_set_gathered: no full volume bound");
    e->gathered = gathered != 0;
    return VC_OK;
}

int vc_slab_words(const vc_engine* e, uint64_t* n_words) {
    if (!e || !n_words) return VC_ERR_ARG;
    *n_words = (uint64_t)e->slab_words;
    return VC_OK;
}

int vc_upload_volumes(vc_engine* e, const uint32_t* occupied, const uint32_t* seen, uint64_t n_words) {
    if (!e) return VC_ERR_ARG;
    if (!occupied || !seen) return fail(e, VC_ERR_ARG, "vc_upload_volumes: null buffer");
    if (n_words != (uint64_t)e->slab_words) return fail(e, VC_ERR_ARG, "vc_upload_volumes: got %llu words, slab has %lld", (unsigned long long)n_words, e->slab_words);
    if (bind_device(e)) return VC_ERR_CUDA;
    if (ensure_volumes(e)) return VC_ERR_CUDA;
    e->reset_pending = false;  // overwritten entirely
    e->flags_valid = false;
    VC_CUDA(e, cudaMemcpyAsync(e->occ_slab(), occupied, n_words * 4, cudaMemcpyHostToDevice, e->stream));
    VC_CUDA(e, cudaMemcpyAsync(e->seen_slab(), seen, n_words * 4, cudaMemcpyHostToDevice, e->stream));
    // padding cleared; [4] counts the words that hold a voxel which is carved but unseen (the reference would still mark such a
    // voxel seen, VoxelCarving.cpp:54, so vc_carve must not skip it: see carve_unseen_begin)
    VC_CUDA(e, cudaMemsetAsync(e->d_scalars + 4, 0, sizeof(unsigned long long), e->stream));
    vc_clear_padding_kernel<<<(unsigned)((e->slab_words + 255) / 256), 256, 0, e->stream>>>(e->occ_slab(), e->seen_slab(), e->slab_words, e->Wx, e->g.X, e->d_scalars + 4);
    VC_CUDA(e, cudaGetLastError());
    unsigned long long n_bad = 0;
    VC_CUDA(e, cudaMemcpyAsync(&n_bad, e->d_scalars + 4, sizeof n_bad, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    e->carved_implies_seen = n_bad == 0;
    e->gathered = false; e->halo_lo = e->halo_hi = false; e->have_colors = false; e->have_mc = false;
    return VC_OK;
}

static int download_words(vc_engine* e, const uint32_t* d, uint32_t* words, uint64_t n_words) {
    if (!words) return fail(e, VC_ERR_ARG, "download: null buffer");
    if (n_words < (uint64_t)e->slab_words) return fail(e, VC_ERR_CAPACITY, "download: buffer holds %llu words, slab has %lld", (unsigned long long)n_words, e->slab_words);
    if (bind_device(e)) return VC_ERR_CUDA;
    if (materialize_reset(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaMemcpyAsync(words, d, e->slab_words * 4, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}
int vc_download_occupied(vc_engine* e, uint32_t* words, uint64_t n_words) { return e ? download_words(e, e->occ_slab(), words, n_words) : VC_ERR_ARG; }
int vc_download_seen(vc_engine* e, uint32_t* words, uint64_t n_words) { return e ? download_words(e, e->seen_slab(), words, n_words) : VC_ERR_ARG; }

int vc_count_occupied(vc_engine* e, uint64_t* n_occupied, uint64_t* n_seen) {
    if (!e || !n_occupied || !n_seen) return VC_ERR_ARG;
    if (bind_device(e)) return VC_ERR_CUDA;
    if (materialize_reset(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaMemsetAsync(e->d_scalars + 3, 0, 2 * sizeof(unsigned long long), e->stream));
    vc_popcount_kernel<<<148 * 8, 256, 0, e->stream>>>(e->occ_slab(), e->seen_slab(), e->slab_words, e->d_scalars + 3);
    VC_CUDA(e, cudaGetLastError());
    unsigned long long h[2];
    VC_CUDA(e, cudaMemcpyAsync(h, e->d_scalars + 3, sizeof h, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    *n_occupied = h[0];
    *n_seen = h[1];
    return VC_OK;
}

// neighbour planes z_begin-1 and z_end must be addressable unless they lie outside the grid
static int need_halo(vc_engine* e, const char* who) {
    if (e->whole_grid() || (e->d_occ_full && e->gathered)) return VC_OK;
    if ((e->g.z_begin == 0 || e->halo_lo) && (e->g.z_end == e->g.Z || e->halo_hi)) return VC_OK;
    return fail(e, VC_ERR_STATE, "%s: slab [%d,%d) of Z=%d needs its neighbour planes: exchange the one-plane halos (vc_exchange_halos / "
                "vc_exchange_halos_peer / vc_import_halo), or gather the whole grid (vc_gather, or an external all-gather + vc_set_gathered(1))",
                who, e->g.z_begin, e->g.z_end, e->g.Z);
}

// The surface records of the slab (occupied & !isInner, ascending flatten index) into d_color_idx / n_surface: a counting
// pass, a scan of the block counts, and an emitting pass.  Clears have_colors first; the caller sets it once its colours are in.
static int build_surface_records(vc_engine* e, const char* who) {
    const long long n = e->slab_words;
    if (n > 0x7fffffffLL) return fail(e, VC_ERR_ARG, "%s: slab of %lld words too large", who, n);
    if (e->nz > 65535) return fail(e, VC_ERR_ARG, "%s: slab of %d planes too deep (grid dimension limit 65535)", who, e->nz);
    const unsigned chunks = (unsigned)((e->plane_words + 1023) / 1024);  // blocks of vc_surface_pass_kernel per plane
    const int nb = (int)(chunks * (unsigned)e->nz);
    const dim3 sgrid(chunks, (unsigned)e->nz);
    if (!e->d_block_sums) VC_CUDA(e, cudaMalloc(&e->d_block_sums, ((size_t)nb + 1) * sizeof(unsigned long long)));
    e->have_colors = false;
    e->n_surface = 0;
    const VcVolView g = vol_view(e);
    vc_surface_pass_kernel<false><<<sgrid, 256, 0, e->stream>>>(g, e->g.z_begin, (unsigned)e->plane_words, e->d_block_sums, nullptr);
    vc_scan_sums_kernel<<<1, 1024, 0, e->stream>>>(e->d_block_sums, nb, e->d_block_sums + nb);
    VC_CUDA(e, cudaGetLastError());
    unsigned long long total = 0;
    VC_CUDA(e, cudaMemcpyAsync(&total, e->d_block_sums + nb, sizeof total, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    if (total > 0xffffffffull) return fail(e, VC_ERR_CAPACITY, "%s: %llu surface voxels exceed 32-bit offsets", who, total);
    e->n_surface = total;
    if (total) {
        if (total > e->color_capacity) {
            free_color(e);
            e->n_surface = total;
            VC_CUDA(e, cudaMalloc(&e->d_color_idx, total * sizeof(unsigned long long)));
            VC_CUDA(e, cudaMalloc(&e->d_color_rgbn, total * sizeof(uchar4)));
            e->color_capacity = total;
        }
        vc_surface_pass_kernel<true><<<sgrid, 256, 0, e->stream>>>(g, e->g.z_begin, (unsigned)e->plane_words, e->d_block_sums, e->d_color_idx);
    }
    return VC_OK;
}

static VcColorParams color_params(const vc_engine* e, int color_mode) {
    VcColorParams p{};
    p.images = e->d_images;
    p.idx_out = e->d_color_idx; p.rgbn_out = e->d_color_rgbn;
    p.X = e->g.X; p.Y = e->g.Y; p.Wx = e->Wx; p.z_begin = e->g.z_begin;
    p.W = e->W; p.H = e->H; p.V = e->V;
    p.s = e->g.voxel_size;
    p.mode = color_mode;
    p.n_surface = e->n_surface;
    p.gview = e->d_view64; p.gcam = e->d_cam;
    return p;
}

int vc_color(vc_engine* e, int32_t color_mode) {
    if (!e) return VC_ERR_ARG;
    PhaseRange nvtx("Coloring");
    if (color_mode != VC_COLOR_CLOSEST && color_mode != VC_COLOR_AVG) return fail(e, VC_ERR_ARG, "vc_color: mode must be 1 (closest) or 2 (average), got %d", color_mode);
    if (e->V == 0 || !e->d_images) return fail(e, VC_ERR_STATE, "vc_color: views and images must be set first");
    if (!e->have_M) return fail(e, VC_ERR_STATE, "vc_color: vc_set_views was given M = NULL (camera translations are needed for the depth)");
    int rc = need_halo(e, "vc_color");
    if (rc) return rc;
    if (bind_device(e)) return VC_ERR_CUDA;
    rc = materialize_reset(e);
    if (rc) return rc;
    const bool global_views = e->V > VC_MAX_VIEWS;  // one pass over every group: P and camera from global memory
    if (!global_views) { rc = ensure_constants(e); if (rc) return rc; }
    rc = build_surface_records(e, "vc_color");
    if (rc) return rc;
    if (e->n_surface) {
        const VcColorParams p = color_params(e, color_mode);
        const unsigned cgrid = (unsigned)((e->n_surface + 255) / 256);
        if (global_views) {
            if (color_mode == VC_COLOR_CLOSEST) vc_surface_color_kernel<1, true><<<cgrid, 256, 0, e->stream>>>(p);
            else vc_surface_color_kernel<2, true><<<cgrid, 256, 0, e->stream>>>(p);
            VC_CUDA(e, cudaGetLastError());
        } else {
            if (color_mode == VC_COLOR_CLOSEST) vc_surface_color_kernel<1><<<cgrid, 256, 0, e->stream>>>(p);
            else vc_surface_color_kernel<2><<<cgrid, 256, 0, e->stream>>>(p);
            VC_CUDA(e, cudaGetLastError());
            rc = constants_used(e);
            if (rc) return rc;
        }
    }
    e->have_colors = true;
    return VC_OK;
}

// Depth buffers of vc_color_visible cover as many views at a time as fit this budget (at least one view).  Every pair is
// splatted and observed exactly once whatever the chunk, so the records do not depend on it; a chunk only bounds the memory.
#define VC_VIS_ZBUF_BUDGET (256ull << 20)

int vc_color_visible(vc_engine* e, int32_t color_mode, float tolerance) {
    if (!e) return VC_ERR_ARG;
    PhaseRange nvtx("Coloring");
    // every refusal before any state changes: the previous colour records stay as they were
    if (color_mode != VC_COLOR_CLOSEST && color_mode != VC_COLOR_AVG) return fail(e, VC_ERR_ARG, "vc_color_visible: mode must be 1 (closest) or 2 (average), got %d", color_mode);
    if (!(tolerance >= 0.0f)) return fail(e, VC_ERR_ARG, "vc_color_visible: tolerance must be >= 0 (voxel sizes), got %g", (double)tolerance);
    if (!e->whole_grid()) return fail(e, VC_ERR_STATE, "vc_color_visible: whole-grid engines only (slab [%d,%d) of Z=%d: occluders in other slabs are unknown)", e->g.z_begin, e->g.z_end, e->g.Z);
    if (e->V == 0 || !e->d_images) return fail(e, VC_ERR_STATE, "vc_color_visible: views and images must be set first");
    if (!e->have_M) return fail(e, VC_ERR_STATE, "vc_color_visible: vc_set_views was given M = NULL (camera translations are needed for the depth)");
    if (bind_device(e)) return VC_ERR_CUDA;
    int rc = materialize_reset(e);
    if (rc) return rc;
    const bool global_views = e->V > VC_MAX_VIEWS;
    if (!global_views) { rc = ensure_constants(e); if (rc) return rc; }
    rc = build_surface_records(e, "vc_color_visible");
    if (rc) return rc;
    const unsigned long long total = e->n_surface;
    if (total) {
        const size_t view_px = (size_t)e->W * e->H;
        const unsigned long long vis_words = (total + 31) / 32;
        const size_t vis_bytes = (size_t)vis_words * 4 * e->V;
        const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)e->V, VC_VIS_ZBUF_BUDGET / (view_px * 4)));
        void* sc = nullptr;
        rc = ensure_scratch(e, vis_bytes + (size_t)chunk * view_px * 4, &sc);
        if (rc) return rc;
        VcVisParams vp{};
        vp.idx = e->d_color_idx; vp.view = e->d_view64;
        vp.vis = (uint32_t*)sc; vp.zbuf = (uint32_t*)((char*)sc + vis_bytes);
        vp.n_surface = total; vp.vis_words = vis_words;
        vp.X = e->g.X; vp.Y = e->g.Y; vp.W = e->W; vp.H = e->H;
        vp.s = e->g.voxel_size;
        vp.tau = tolerance * e->g.voxel_size;  // fl(tolerance * s)
        const unsigned bx = (unsigned)((total + 255) / 256);
        for (int v0 = 0; v0 < e->V; v0 += chunk) {
            const int nv = std::min(chunk, e->V - v0);
            vp.v0 = v0;
            // 0xffffffff is above the bits of every key (+inf included) and is read nowhere: a pair reads its own centre pixel
            VC_CUDA(e, cudaMemsetAsync(vp.zbuf, 0xff, (size_t)nv * view_px * 4, e->stream));
            vc_vis_splat_kernel<<<dim3(bx, (unsigned)nv), 256, 0, e->stream>>>(vp);
            vc_vis_observe_kernel<<<dim3(bx, (unsigned)nv), 256, 0, e->stream>>>(vp);
            VC_CUDA(e, cudaGetLastError());
        }
        VcColorParams p = color_params(e, color_mode);
        p.vis = vp.vis; p.vis_words = vis_words;
        if (global_views) {
            if (color_mode == VC_COLOR_CLOSEST) vc_surface_color_kernel<1, true, true><<<bx, 256, 0, e->stream>>>(p);
            else vc_surface_color_kernel<2, true, true><<<bx, 256, 0, e->stream>>>(p);
            VC_CUDA(e, cudaGetLastError());
        } else {
            if (color_mode == VC_COLOR_CLOSEST) vc_surface_color_kernel<1, false, true><<<bx, 256, 0, e->stream>>>(p);
            else vc_surface_color_kernel<2, false, true><<<bx, 256, 0, e->stream>>>(p);
            VC_CUDA(e, cudaGetLastError());
            rc = constants_used(e);
            if (rc) return rc;
        }
    }
    e->have_colors = true;
    return VC_OK;
}

int vc_surface_count(vc_engine* e, uint64_t* n) {
    if (!e || !n) return VC_ERR_ARG;
    if (!e->have_colors) return fail(e, VC_ERR_STATE, "vc_surface_count: run vc_color first");
    *n = e->n_surface;
    return VC_OK;
}

int vc_download_colors(vc_engine* e, uint64_t* idx, uint8_t* rgbn, uint64_t capacity) {
    if (!e) return VC_ERR_ARG;
    if (!e->have_colors) return fail(e, VC_ERR_STATE, "vc_download_colors: run vc_color first");
    if (capacity < e->n_surface) return fail(e, VC_ERR_CAPACITY, "vc_download_colors: capacity %llu < %llu surface voxels", (unsigned long long)capacity, e->n_surface);
    if (e->n_surface == 0) return VC_OK;
    if (!idx || !rgbn) return fail(e, VC_ERR_ARG, "vc_download_colors: null buffer");
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaMemcpyAsync(idx, e->d_color_idx, e->n_surface * 8, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaMemcpyAsync(rgbn, e->d_color_rgbn, e->n_surface * 4, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

int vc_mc_classify(vc_engine* e) {
    if (!e) return VC_ERR_ARG;
    PhaseRange nvtx("MarchingCubes");
    int rc = need_halo(e, "vc_mc_classify");
    if (rc) return rc;
    if (bind_device(e)) return VC_ERR_CUDA;
    rc = materialize_reset(e);
    if (rc) return rc;
    // cells whose lower plane z is in [z_begin, z_end), plus z = -1 on the first slab (MarchingCubes.cpp:14)
    const int cz_begin = e->g.z_begin == 0 ? -1 : e->g.z_begin;
    const int n_cz = e->g.z_end - cz_begin;
    const int Cw = (e->g.X + 1 + 31) / 32;
    const long long n = (long long)n_cz * (e->g.Y + 1) * Cw;
    VC_CUDA(e, cudaMemsetAsync(e->d_hist, 0, 257 * sizeof(unsigned long long), e->stream));
    const long long n_tasks = (long long)n_cz * ((e->g.Y + 1 + VC_MC_ROWS - 1) / VC_MC_ROWS) * ((Cw + 31) / 32);  // one warp each
    long long blocks = (n_tasks + 7) / 8;
    if (blocks > (long long)e->sm_count * 4) blocks = (long long)e->sm_count * 4;  // persistent: warps pull tasks from a counter
    (void)n;
    VcMcFlags mf{};
    mf.enabled = (e->flags_valid && e->d_brick_flags && !e->reset_pending) ? 1 : 0;
    mf.brick_flags = e->d_brick_flags; mf.super_flags = e->d_super_flags;
    const BrickGeom b = brick_geom(e, e->nz);
    mf.nby = b.nby; mf.pbx = b.sbx; mf.pby = b.sby;
    mf.z_begin = e->g.z_begin; mf.z_end = e->g.z_end;
    vc_mc_classify_kernel<<<(unsigned)blocks, 256, 0, e->stream>>>(vol_view(e), cz_begin, n_cz, Cw, e->d_hist, mf);
    VC_CUDA(e, cudaGetLastError());
    e->have_mc = true;
    return VC_OK;
}

int vc_download_mc(vc_engine* e, uint64_t hist256[256], uint64_t* n_active, uint64_t* n_triangles) {
    if (!e || !hist256 || !n_active || !n_triangles) return VC_ERR_ARG;
    if (!e->have_mc) return fail(e, VC_ERR_STATE, "vc_download_mc: run vc_mc_classify first");
    if (bind_device(e)) return VC_ERR_CUDA;
    unsigned long long h[256];
    VC_CUDA(e, cudaMemcpyAsync(h, e->d_hist, sizeof h, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    uint64_t act = 0, tris = 0;
    for (int i = 0; i < 256; i++) {
        hist256[i] = h[i];
        int nt = 0;
        for (int k = 0; k < 16 && VC_TRI_TABLE_HEX[i * 16 + k] != 'f'; k++) nt++;
        tris += h[i] * (uint64_t)(nt / 3);  // triTable row length / 3 (MarchingCubes.h:503)
        if (i != 0 && i != 255) act += h[i];  // edgeTable[idx] != 0 (MarchingCubes.h:486)
    }
    *n_active = act;
    *n_triangles = tris;
    return VC_OK;
}

int vc_get_stats(vc_engine* e, vc_stats* out) {
    if (!e || !out) return VC_ERR_ARG;
    if (bind_device(e)) return VC_ERR_CUDA;
    if (e->stats.last_carve_ms < 0.0 && e->stats.carve_launches > 0) {
        VC_CUDA(e, cudaEventSynchronize(e->ev1));
        float ms = 0.f;
        VC_CUDA(e, cudaEventElapsedTime(&ms, e->ev0, e->ev1));
        e->stats.last_carve_ms = ms;
        e->stats.last_classify_ms = 0.0;
        if (e->have_mid) {
            VC_CUDA(e, cudaEventElapsedTime(&ms, e->ev0, e->evm));
            e->stats.last_classify_ms = ms;
        }
    }
    *out = e->stats;
    return VC_OK;
}

int vc_measure_peaks(int32_t device, double* ffma_tflops, double* dfma_tflops) {
    if (!ffma_tflops || !dfma_tflops) return VC_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_measure_peaks: cudaSetDevice(%d) failed", device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_measure_peaks: no device properties");
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    void* d = nullptr;
    cudaEvent_t a, b;
    if (cudaMalloc(&d, (size_t)blocks * threads * 8) != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_measure_peaks: cudaMalloc failed");
    cudaEventCreate(&a); cudaEventCreate(&b);
    double best[2] = {0, 0};
    for (int which = 0; which < 2; which++) {
        const int iters = which == 0 ? 1 << 15 : 1 << 13;
        for (int rep = 0; rep < 6; rep++) {
            cudaEventRecord(a);
            if (which == 0) vc_fma_peak_kernel<float><<<blocks, threads>>>((float*)d, iters, 1.0000001f, 1e-7f);
            else vc_fma_peak_kernel<double><<<blocks, threads>>>((double*)d, iters, 1.0000001, 1e-7);
            cudaEventRecord(b);
            cudaEventSynchronize(b);
            float ms = 0;
            cudaEventElapsedTime(&ms, a, b);
            const double tf = 2.0 * 8.0 * iters * (double)blocks * threads / (ms * 1e-3) / 1e12;
            if (rep > 0 && tf > best[which]) best[which] = tf;
        }
    }
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(d);
    cudaError_t s = cudaGetLastError();
    if (s != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_measure_peaks: %s", cudaGetErrorString(s));
    *ffma_tflops = best[0];
    *dfma_tflops = best[1];
    return VC_OK;
}

static int load_mc_tables(vc_engine* e);

static int dense_ready(vc_engine* e, const char* who, bool need_data) {
    if (!e->whole_grid()) return fail(e, VC_ERR_STATE, "%s: the dense Model needs the whole grid on one engine", who);
    if (bind_device(e)) return VC_ERR_CUDA;
    const size_t n = (size_t)e->g.X * e->g.Y * e->g.Z;
    if (!e->d_dense) VC_CUDA(e, cudaMalloc(&e->d_dense, n * sizeof(float4)));
    if (need_data && !e->have_dense) return fail(e, VC_ERR_STATE, "%s: no dense Model yet (vc_dense_upload / vc_dense_from_volumes)", who);
    return load_mc_tables(e);
}

static int load_mc_tables(vc_engine* e) {
    static std::mutex m;
    static bool tables[64] = {};
    std::lock_guard<std::mutex> lk(m);
    if (!tables[e->g.device & 63]) {  // triTable -> constant memory, once per device
        signed char tri[256][16];
        unsigned char ntri[256];
        for (int i = 0; i < 256; i++) {
            int k = 0;
            for (; k < 16; k++) {
                const char c = VC_TRI_TABLE_HEX[i * 16 + k];
                tri[i][k] = c == 'f' ? -1 : (signed char)(c <= '9' ? c - '0' : c - 'a' + 10);
            }
            int nt = 0;
            while (nt < 16 && tri[i][nt] != -1) nt++;
            ntri[i] = (unsigned char)(nt / 3);
        }
        VC_CUDA(e, cudaMemcpyToSymbol(c_tri, tri, sizeof tri));
        VC_CUDA(e, cudaMemcpyToSymbol(c_ntri, ntri, sizeof ntri));
        tables[e->g.device & 63] = true;
    }
    return VC_OK;
}

int vc_dense_upload(vc_engine* e, const float* rgba) {
    if (!e) return VC_ERR_ARG;
    if (!rgba) return fail(e, VC_ERR_ARG, "vc_dense_upload: null buffer");
    int rc = dense_ready(e, "vc_dense_upload", false);
    if (rc) return rc;
    const size_t n = (size_t)e->g.X * e->g.Y * e->g.Z;
    VC_CUDA(e, cudaMemcpyAsync(e->d_dense, rgba, n * sizeof(float4), cudaMemcpyHostToDevice, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    e->have_dense = true; e->have_mesh = false;
    return VC_OK;
}

int vc_dense_from_volumes(vc_engine* e, int32_t apply_colors, int32_t handle_unseen) {
    if (!e) return VC_ERR_ARG;
    int rc = dense_ready(e, "vc_dense_from_volumes", false);
    if (rc) return rc;
    if (apply_colors && !e->have_colors) return fail(e, VC_ERR_STATE, "vc_dense_from_volumes: apply_colors needs a preceding vc_color");
    rc = materialize_reset(e);
    if (rc) return rc;
    const size_t n = (size_t)e->g.X * e->g.Y * e->g.Z;
    VcDense d{e->d_dense, e->g.X, e->g.Y, e->g.Z};
    vc_dense_base_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(d, e->occ_slab(), e->Wx);
    if (apply_colors && e->n_surface)
        vc_dense_colors_kernel<<<(unsigned)((e->n_surface + 255) / 256), 256, 0, e->stream>>>(d, e->d_color_idx, e->d_color_rgbn, e->n_surface);
    if (handle_unseen) vc_dense_unseen_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(d, e->seen_slab(), e->Wx);
    VC_CUDA(e, cudaGetLastError());
    e->have_dense = true; e->have_mesh = false;
    return VC_OK;
}

int vc_dense_apply_carved(vc_engine* e) {
    if (!e) return VC_ERR_ARG;
    int rc = dense_ready(e, "vc_dense_apply_carved", true);
    if (rc) return rc;
    rc = materialize_reset(e);
    if (rc) return rc;
    const size_t n = (size_t)e->g.X * e->g.Y * e->g.Z;
    VcDense d{e->d_dense, e->g.X, e->g.Y, e->g.Z};
    vc_dense_carved_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(d, e->occ_slab(), e->Wx);
    VC_CUDA(e, cudaGetLastError());
    e->have_mesh = false;
    return VC_OK;
}

int vc_dense_closure(vc_engine* e, int32_t kernel_size) {
    if (!e) return VC_ERR_ARG;
    PhaseRange nvtx("PostProcessing");
    if (kernel_size < 1 || kernel_size % 2 != 1) return fail(e, VC_ERR_ARG, "Invalid kernel size for post processing, skipping...");  // Postprocessing3d.cpp:8-11
    int rc = dense_ready(e, "vc_dense_closure", true);
    if (rc) return rc;
    const size_t n = (size_t)e->g.X * e->g.Y * e->g.Z;
    if (!e->d_dense_tmp) VC_CUDA(e, cudaMalloc(&e->d_dense_tmp, n * sizeof(float4)));
    VcDense d{e->d_dense, e->g.X, e->g.Y, e->g.Z};
    vc_closure_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(d, e->d_dense_tmp, (kernel_size - 1) / 2);
    VC_CUDA(e, cudaGetLastError());
    std::swap(e->d_dense, e->d_dense_tmp);
    e->have_mesh = false;
    return VC_OK;
}

int vc_dense_download(vc_engine* e, float* rgba) {
    if (!e) return VC_ERR_ARG;
    if (!rgba) return fail(e, VC_ERR_ARG, "vc_dense_download: null buffer");
    int rc = dense_ready(e, "vc_dense_download", true);
    if (rc) return rc;
    const size_t n = (size_t)e->g.X * e->g.Y * e->g.Z;
    VC_CUDA(e, cudaMemcpyAsync(rgba, e->d_dense, n * sizeof(float4), cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

// exclusive scan of the per-column triangle counts into offsets (in place), then room for the triangles in the grow-only mesh
// buffers.  Refused (VC_ERR_CAPACITY) before anything of the previous mesh is touched when the offsets would overflow.
static int scan_mesh_counts(vc_engine* e, const char* who, uint32_t* d_counts, unsigned long long* d_sums, long long ncol, int nb,
                            unsigned long long* total_out) {
    vc_scan_block_kernel<<<nb, VC_SCAN_BLOCK, 0, e->stream>>>(d_counts, d_counts, d_sums, ncol);
    vc_scan_sums_kernel<<<1, 1024, 0, e->stream>>>(d_sums, nb, d_sums + nb);
    vc_scan_add_kernel<<<nb, VC_SCAN_BLOCK, 0, e->stream>>>(d_counts, d_sums, ncol);
    VC_CUDA(e, cudaGetLastError());
    unsigned long long total = 0;
    VC_CUDA(e, cudaMemcpyAsync(&total, d_sums + nb, sizeof total, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    if (total > 0xffffffffull) return fail(e, VC_ERR_CAPACITY, "%s: %llu triangles exceed 32-bit offsets", who, total);
    if (total > e->mesh_capacity) {  // triangle buffers are grow-only
        e->have_mesh = false;
        e->mesh_version++;
        cudaFree(e->d_mesh_verts); cudaFree(e->d_mesh_rgb); e->d_mesh_verts = nullptr; e->d_mesh_rgb = nullptr; e->mesh_capacity = 0;
        VC_CUDA(e, cudaMalloc(&e->d_mesh_verts, total * 9 * sizeof(float)));
        VC_CUDA(e, cudaMalloc(&e->d_mesh_rgb, total * 3 * sizeof(uint32_t)));
        e->mesh_capacity = total;
    }
    *total_out = total;
    return VC_OK;
}

int vc_mc_mesh(vc_engine* e, float threshold, uint64_t* n_triangles) {
    if (!e || !n_triangles) return VC_ERR_ARG;
    PhaseRange nvtx("MarchingCubes");
    int rc = dense_ready(e, "vc_mc_mesh", true);
    if (rc) return rc;
    const long long ncol = (long long)(e->g.X + 1) * (e->g.Y + 1);
    if (ncol > 0x7fffffffLL) return fail(e, VC_ERR_ARG, "vc_mc_mesh: grid too large");
    const int nb = (int)((ncol + VC_SCAN_BLOCK - 1) / VC_SCAN_BLOCK);
    void* sc = nullptr;
    const size_t counts_bytes = ((size_t)ncol * 4 + 15) / 16 * 16;
    rc = ensure_scratch(e, counts_bytes + ((size_t)nb + 1) * sizeof(unsigned long long), &sc);
    if (rc) return rc;
    uint32_t* d_counts = (uint32_t*)sc;
    unsigned long long* d_sums = (unsigned long long*)((char*)sc + counts_bytes);
    VcDense d{e->d_dense, e->g.X, e->g.Y, e->g.Z};
    vc_mc_count_kernel<<<(unsigned)((ncol + 127) / 128), 128, 0, e->stream>>>(d, threshold, d_counts);
    unsigned long long total = 0;
    rc = scan_mesh_counts(e, "vc_mc_mesh", d_counts, d_sums, ncol, nb, &total);
    if (rc) return rc;
    if (total) {
        vc_mc_emit_kernel<<<(unsigned)((ncol + 127) / 128), 128, 0, e->stream>>>(d, threshold, d_counts, e->d_mesh_verts, e->d_mesh_rgb);
        VC_CUDA(e, cudaGetLastError());
    }
    e->n_mesh_tris = total;
    e->have_mesh = true;
    e->mesh_version++;
    *n_triangles = total;
    return VC_OK;
}

int vc_mesh_from_volumes(vc_engine* e, int32_t apply_colors, int32_t handle_unseen, int32_t closure_k, float threshold, uint64_t* n_triangles) {
    if (!e || !n_triangles) return VC_ERR_ARG;
    PhaseRange nvtx("MarchingCubes");
    if (closure_k < 0 || closure_k > VC_MESH_MAX_CLOSURE || (closure_k != 0 && closure_k % 2 != 1))
        return fail(e, VC_ERR_ARG, "vc_mesh_from_volumes: closure kernel size must be 0 (none) or odd in [1, %d], got %d", VC_MESH_MAX_CLOSURE, closure_k);
    if (!e->whole_grid()) return fail(e, VC_ERR_STATE, "vc_mesh_from_volumes: meshing needs the whole grid on one engine");
    if (apply_colors && !e->have_colors) return fail(e, VC_ERR_STATE, "vc_mesh_from_volumes: apply_colors needs a vc_color of the current volumes");
    const long long ncol = (long long)(e->g.X + 1) * (e->g.Y + 1);
    if (ncol > 0x7fffffffLL) return fail(e, VC_ERR_ARG, "vc_mesh_from_volumes: grid too large");
    if (bind_device(e)) return VC_ERR_CUDA;
    int rc = load_mc_tables(e);
    if (rc) return rc;
    rc = materialize_reset(e);
    if (rc) return rc;
    // alphas are 0 or 1: any other threshold puts every corner on one side (no triangles)
    if (!(threshold > 0.f && threshold <= 1.f)) {
        e->n_mesh_tris = 0;
        e->have_mesh = true;
        e->mesh_version++;
        *n_triangles = 0;
        return VC_OK;
    }
    const int s = closure_k > 0 ? (closure_k - 1) / 2 : 0;
    const bool colors = apply_colors && e->n_surface > 0;
    const long long n_rows = (long long)e->g.Y * e->g.Z;
    const int nb = (int)((ncol + VC_SCAN_BLOCK - 1) / VC_SCAN_BLOCK);
    // scratch: column counts | scan block sums | record row offsets (colours) | dilated occupancy (closure)
    const size_t counts_bytes = ((size_t)ncol * 4 + 15) / 16 * 16;
    const size_t sums_bytes = (((size_t)nb + 1) * sizeof(unsigned long long) + 15) / 16 * 16;
    const size_t rows_bytes = colors ? ((size_t)(n_rows + 1) * 4 + 15) / 16 * 16 : 0;
    const size_t dil_bytes = s > 0 ? (size_t)e->slab_words * 4 : 0;
    void* sc = nullptr;
    rc = ensure_scratch(e, counts_bytes + sums_bytes + rows_bytes + dil_bytes, &sc);
    if (rc) return rc;
    uint32_t* d_counts = (uint32_t*)sc;
    unsigned long long* d_sums = (unsigned long long*)((char*)sc + counts_bytes);
    uint32_t* d_rows = (uint32_t*)((char*)sc + counts_bytes + sums_bytes);
    uint32_t* d_dil = (uint32_t*)((char*)sc + counts_bytes + sums_bytes + rows_bytes);
    VcMeshSrc m{};
    m.occ = e->occ_slab(); m.seen = e->seen_slab();
    m.X = e->g.X; m.Y = e->g.Y; m.Z = e->g.Z; m.Wx = e->Wx;
    m.unseen = handle_unseen ? 1 : 0;
    m.s = s;
    if (colors) {
        m.rec_idx = e->d_color_idx; m.rec_rgbn = e->d_color_rgbn; m.row_start = d_rows;
        vc_record_rows_kernel<<<(unsigned)((n_rows + 1 + 255) / 256), 256, 0, e->stream>>>(e->d_color_idx, (uint32_t)e->n_surface, e->g.X, n_rows, d_rows);
    }
    if (s > 0) {
        int zchunk = 64;  // planes per thread (each chunk re-reads 2s planes of its neighbours)
        while ((long long)e->g.Y * e->Wx * ((e->g.Z + zchunk - 1) / zchunk) > 0x7fffffffLL) zchunk *= 2;
        const long long n_threads = (long long)e->g.Y * e->Wx * ((e->g.Z + zchunk - 1) / zchunk);
        vc_dilate_kernel<<<(unsigned)((n_threads + 255) / 256), 256, 0, e->stream>>>(m, zchunk, d_dil);
        m.dil = d_dil;
    }
    vc_mesh_count_kernel<<<(unsigned)((ncol + 255) / 256), 256, 0, e->stream>>>(m, d_counts);
    unsigned long long total = 0;
    rc = scan_mesh_counts(e, "vc_mesh_from_volumes", d_counts, d_sums, ncol, nb, &total);
    if (rc) return rc;
    if (total) {
        vc_mesh_emit_kernel<<<(unsigned)((ncol + 127) / 128), 128, 0, e->stream>>>(m, d_counts, e->d_mesh_verts);
        vc_mesh_color_kernel<<<(unsigned)((total + 255) / 256), 256, 0, e->stream>>>(m, e->d_mesh_verts, total, e->d_mesh_rgb);
        VC_CUDA(e, cudaGetLastError());
    }
    e->n_mesh_tris = total;
    e->have_mesh = true;
    e->mesh_version++;
    *n_triangles = total;
    return VC_OK;
}

int vc_download_mesh(vc_engine* e, float* verts, uint32_t* rgb, uint64_t capacity_triangles) {
    if (!e) return VC_ERR_ARG;
    if (!e->have_mesh) return fail(e, VC_ERR_STATE, "vc_download_mesh: run vc_mc_mesh first");
    if (capacity_triangles < e->n_mesh_tris) return fail(e, VC_ERR_CAPACITY, "vc_download_mesh: capacity %llu < %llu triangles", (unsigned long long)capacity_triangles, e->n_mesh_tris);
    if (e->n_mesh_tris == 0) return VC_OK;
    if (!verts || !rgb) return fail(e, VC_ERR_ARG, "vc_download_mesh: null buffer");
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaMemcpyAsync(verts, e->d_mesh_verts, e->n_mesh_tris * 9 * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaMemcpyAsync(rgb, e->d_mesh_rgb, e->n_mesh_tris * 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

// Length pass and scan of a text's s.n_lines (>= 1) lines: d_lens (n_lines u32) becomes the lines' offsets inside their scan
// block, d_sums (nb + 1 u64) the blocks' offsets with the total at [nb].  Ends in a synchronisation of `st`.
static cudaError_t text_scan(const VcTextSrc& s, uint32_t* d_lens, unsigned long long* d_sums, cudaStream_t st, unsigned long long* total) {
    const int nb = (int)((s.n_lines + VC_SCAN_BLOCK - 1) / VC_SCAN_BLOCK);
    vc_text_len_kernel<<<(unsigned)((s.n_lines + 255) / 256), 256, 0, st>>>(s, d_lens);
    vc_scan_block_kernel<<<nb, VC_SCAN_BLOCK, 0, st>>>(d_lens, d_lens, d_sums, (long long)s.n_lines);
    vc_scan_sums_kernel<<<1, 1024, 0, st>>>(d_sums, nb, d_sums + nb);
    cudaError_t r = cudaGetLastError();
    if (r == cudaSuccess) r = cudaMemcpyAsync(total, d_sums + nb, sizeof *total, cudaMemcpyDeviceToHost, st);
    if (r == cudaSuccess) r = cudaStreamSynchronize(st);
    return r;
}
// the lines themselves, at byte `base` of d_text onwards (after text_scan on the same buffers)
static cudaError_t text_emit(const VcTextSrc& s, const uint32_t* d_offs, const unsigned long long* d_sums, unsigned long long base, char* d_text,
                             cudaStream_t st) {
    const int nb = (int)((s.n_lines + VC_SCAN_BLOCK - 1) / VC_SCAN_BLOCK);
    cudaError_t r = cudaFuncSetAttribute(vc_text_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, VC_TEXT_SMEM);
    if (r != cudaSuccess) return r;
    vc_text_emit_kernel<<<nb, VC_SCAN_BLOCK, VC_TEXT_SMEM, st>>>(s, d_offs, d_sums, base, d_text);
    return cudaGetLastError();
}

int vc_mesh_format_off(vc_engine* e, float scale, float tx, float ty, float tz, uint64_t* n_bytes) {
    if (!e || !n_bytes) return VC_ERR_ARG;
    if (!e->have_mesh) return fail(e, VC_ERR_STATE, "vc_mesh_format_off: no mesh on the device (vc_mc_mesh / vc_mesh_from_volumes first)");
    const unsigned long long T = e->n_mesh_tris, L = 4 * T;
    if (L > VC_TEXT_MAX_LINES)
        return fail(e, VC_ERR_CAPACITY, "vc_mesh_format_off: %llu triangles make %llu lines, more than the %llu one text takes", T, L, VC_TEXT_MAX_LINES);
    if (bind_device(e)) return VC_ERR_CUDA;
    PhaseRange nvtx("WriteMesh");
    char hdr[64];
    const int hl = snprintf(hdr, sizeof hdr, "OFF\n%llu %llu 0\n", 3 * T, T);
    const VcTextSrc src{nullptr, e->d_mesh_verts, e->d_mesh_rgb, T, L, scale, {tx, ty, tz}};
    const int nb = (int)((L + VC_SCAN_BLOCK - 1) / VC_SCAN_BLOCK);
    const size_t lens_bytes = ((size_t)L * 4 + 15) / 16 * 16;
    unsigned long long body = 0;
    uint32_t* d_lens = nullptr;
    unsigned long long* d_sums = nullptr;
    if (L) {
        void* sc = nullptr;
        int rc = ensure_scratch(e, lens_bytes + ((size_t)nb + 1) * sizeof(unsigned long long), &sc);
        if (rc) return rc;
        d_lens = (uint32_t*)sc;
        d_sums = (unsigned long long*)((char*)sc + lens_bytes);
        VC_CUDA(e, text_scan(src, d_lens, d_sums, e->stream, &body));
    }
    const unsigned long long total = hl + body;
    if (total > e->text_capacity) {  // grow-only; the previous text stays until the new buffer exists
        char* t = nullptr;
        VC_CUDA(e, cudaMalloc(&t, total));
        cudaFree(e->d_text);
        e->d_text = t;
        e->text_capacity = total;
    }
    e->have_text = false;
    VC_CUDA(e, cudaMemcpyAsync(e->d_text, hdr, hl, cudaMemcpyHostToDevice, e->stream));
    if (L) VC_CUDA(e, text_emit(src, d_lens, d_sums, hl, e->d_text, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    e->text_bytes = total;
    e->text_version = e->mesh_version;
    e->have_text = true;
    *n_bytes = total;
    return VC_OK;
}

int vc_download_mesh_off(vc_engine* e, uint64_t offset, void* dst, uint64_t n_bytes) {
    if (!e) return VC_ERR_ARG;
    if (!e->have_text) return fail(e, VC_ERR_STATE, "vc_download_mesh_off: no text formatted (vc_mesh_format_off first)");
    if (e->text_version != e->mesh_version) return fail(e, VC_ERR_STATE, "vc_download_mesh_off: the mesh changed since its text was formatted");
    if (offset > e->text_bytes || n_bytes > e->text_bytes - offset)
        return fail(e, VC_ERR_ARG, "vc_download_mesh_off: bytes [%llu, %llu + %llu) lie past the end of the %llu-byte text", (unsigned long long)offset,
                    (unsigned long long)offset, (unsigned long long)n_bytes, e->text_bytes);
    if (n_bytes == 0) return VC_OK;
    if (!dst) return fail(e, VC_ERR_ARG, "vc_download_mesh_off: null buffer");
    if (bind_device(e)) return VC_ERR_CUDA;
    VC_CUDA(e, cudaMemcpyAsync(dst, e->d_text + offset, n_bytes, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

int vc_format_g(int32_t device, uint64_t n, const float* values, char* text, uint64_t capacity, uint64_t* n_bytes) {
    if (!n_bytes || (n && !values)) return fail(nullptr, VC_ERR_ARG, "vc_format_g: null argument");
    if (n > VC_TEXT_MAX_LINES) return fail(nullptr, VC_ERR_CAPACITY, "vc_format_g: %llu values, more than the %llu lines one text takes", (unsigned long long)n, VC_TEXT_MAX_LINES);
    *n_bytes = 0;
    if (n == 0) return VC_OK;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return fail(nullptr, VC_ERR_CUDA, "vc_format_g: no CUDA device %d; this engine has no CPU fallback", device); }
    const int nb = (int)((n + VC_SCAN_BLOCK - 1) / VC_SCAN_BLOCK);
    float* d_values = nullptr;
    uint32_t* d_lens = nullptr;
    unsigned long long* d_sums = nullptr;
    char* d_text = nullptr;
    unsigned long long total = 0;
    bool room = false;
    cudaError_t s = cudaMalloc(&d_values, n * sizeof(float));
    if (s == cudaSuccess) s = cudaMalloc(&d_lens, n * sizeof(uint32_t));
    if (s == cudaSuccess) s = cudaMalloc(&d_sums, ((size_t)nb + 1) * sizeof(unsigned long long));
    if (s == cudaSuccess) s = cudaMemcpy(d_values, values, n * sizeof(float), cudaMemcpyHostToDevice);
    const VcTextSrc src{d_values, nullptr, nullptr, 0, n, 1.f, {0.f, 0.f, 0.f}};
    if (s == cudaSuccess) s = text_scan(src, d_lens, d_sums, 0, &total);
    if (s == cudaSuccess) {
        *n_bytes = total;
        room = total <= capacity && text;
    }
    if (s == cudaSuccess && room) s = cudaMalloc(&d_text, total);
    if (s == cudaSuccess && room) s = text_emit(src, d_lens, d_sums, 0, d_text, 0);
    if (s == cudaSuccess && room) s = cudaMemcpy(text, d_text, total, cudaMemcpyDeviceToHost);
    cudaFree(d_values); cudaFree(d_lens); cudaFree(d_sums); cudaFree(d_text);
    if (s != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_format_g: %s", cudaGetErrorString(s));
    if (!room) return fail(nullptr, total > capacity ? VC_ERR_CAPACITY : VC_ERR_ARG, "vc_format_g: the text has %llu bytes, the buffer %llu", total,
                           text ? (unsigned long long)capacity : 0ull);
    return VC_OK;
}

int vc_selftest(int32_t device, int32_t which, uint64_t n, uint64_t seed, uint64_t* mismatches, uint64_t* checked) {
    if (!mismatches || !checked || which < 0 || which > 2) return VC_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_selftest: cudaSetDevice(%d) failed", device);
    unsigned long long* d = nullptr;
    if (cudaMalloc(&d, 16) != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_selftest: cudaMalloc failed");
    cudaMemset(d, 0, 16);
    vc_selftest_kernel<<<148 * 8, 256>>>(which, n, seed, d, d + 1);
    unsigned long long h[2] = {0, 0};
    cudaError_t s = cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (s != cudaSuccess) return fail(nullptr, VC_ERR_CUDA, "vc_selftest: %s", cudaGetErrorString(s));
    *mismatches = h[0];
    *checked = h[1];
    return VC_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Multi-GPU: one-plane halos and collectives (SURVEY §8e).  Voxels are independent, so carving needs no exchange; the
// consumers of the grid read one neighbour plane of `occupied` (isInner, Model.h:126-132: z - 1 and z + 1; the cube index,
// MarchingCubes.h:537-552: z + 1).  Engines in one process swap those planes with plain device copies
// (vc_exchange_halos_peer); engines in different processes - one rank per GPU - through NCCL send/recv (vc_exchange_halos);
// vc_gather assembles the whole grid, which only a host-side Model needs.
// NCCL is loaded at run time (dlopen), so libvoxcarve.so has no load-time dependency on it: a process that already
// carries an NCCL (PyTorch ships its own) shares that copy, everything else picks up the system's libnccl.so.2.
// ---------------------------------------------------------------------------------------------
namespace {
struct NcclApi {
    void* handle = nullptr;
    int version = 0;
    decltype(&ncclGetVersion) GetVersion = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclSend) Send = nullptr;
    decltype(&ncclRecv) Recv = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    std::string error;
};
NcclApi g_nccl;
std::mutex g_nccl_mutex;

const NcclApi* load_nccl() {
    std::lock_guard<std::mutex> lk(g_nccl_mutex);
    if (g_nccl.handle) return &g_nccl;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // the copy this process already carries (e.g. PyTorch's), if any
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
    if (!h) { g_nccl.error = std::string("cannot load libnccl.so.2: ") + dlerror(); return nullptr; }
    NcclApi a;
    a.handle = h;
#define VC_NCCL_SYM(field, name)                                                                     \
    a.field = (decltype(a.field))dlsym(h, name);                                                     \
    if (!a.field) { g_nccl.error = std::string("libnccl.so.2 lacks ") + name; dlclose(h); return nullptr; }
    VC_NCCL_SYM(GetVersion, "ncclGetVersion") VC_NCCL_SYM(GetUniqueId, "ncclGetUniqueId") VC_NCCL_SYM(CommInitRank, "ncclCommInitRank")
    VC_NCCL_SYM(CommDestroy, "ncclCommDestroy") VC_NCCL_SYM(GetErrorString, "ncclGetErrorString") VC_NCCL_SYM(GroupStart, "ncclGroupStart")
    VC_NCCL_SYM(GroupEnd, "ncclGroupEnd") VC_NCCL_SYM(Send, "ncclSend") VC_NCCL_SYM(Recv, "ncclRecv")
    VC_NCCL_SYM(AllGather, "ncclAllGather") VC_NCCL_SYM(AllReduce, "ncclAllReduce")
#undef VC_NCCL_SYM
    a.GetVersion(&a.version);
    g_nccl = a;
    return &g_nccl;
}

#define VC_NCCL(e, api, call)                                                                                            \
    do {                                                                                                                 \
        ncclResult_t _r = (call);                                                                                        \
        if (_r != ncclSuccess)                                                                                           \
            return fail((e), VC_ERR_COMM, "%s failed: %s (%s:%d)", #call, (api)->GetErrorString(_r), __FILE__, __LINE__); \
    } while (0)

// first plane of the halo slot `which` (0: plane z_begin - 1, 1: plane z_end), or null when that plane is outside the grid
uint32_t* halo_slot(vc_engine* e, int which) {
    if (which == 0) return e->g.z_begin > 0 ? e->occ_slab() - e->plane_words : nullptr;
    return e->g.z_end < e->g.Z ? e->occ_slab() + e->slab_words : nullptr;
}
}  // namespace

extern "C" {

int vc_alloc_full_volumes(vc_engine* e) {
    if (!e) return VC_ERR_ARG;
    if (bind_device(e)) return VC_ERR_CUDA;
    if (e->d_occ_full_own) return VC_OK;
    const size_t bytes = (size_t)e->g.Z * e->plane_words * 4;
    uint32_t *o = nullptr, *s = nullptr;
    VC_CUDA(e, vol_alloc(e, &o, bytes));
    if (vol_alloc(e, &s, bytes) != cudaSuccess) { vol_free(o); cudaGetLastError(); return fail(e, VC_ERR_CUDA, "vc_alloc_full_volumes: out of device memory (%zu bytes per volume)", bytes); }
    int rc = vc_bind_volumes(e, o, s);  // drops the slab-sized volumes' role; resets the state
    if (rc) { vol_free(o); vol_free(s); return rc; }
    e->d_occ_full_own = o;
    e->d_seen_full_own = s;
    vol_free(e->d_occ_own); vol_free(e->d_seen_own);
    e->d_occ_own = e->d_seen_own = nullptr;
    return VC_OK;
}

int vc_halo_words(const vc_engine* e, uint64_t* n_words) {
    if (!e || !n_words) return VC_ERR_ARG;
    *n_words = (uint64_t)e->plane_words;
    return VC_OK;
}

int vc_export_halo(vc_engine* e, int32_t which, void** d_plane) {
    if (!e || !d_plane || (which != 0 && which != 1)) return VC_ERR_ARG;
    int rc = materialize_reset(e);
    if (rc) return rc;
    *d_plane = which == 0 ? e->occ_slab() : e->occ_slab() + e->slab_words - e->plane_words;
    return VC_OK;
}

int vc_import_halo(vc_engine* e, int32_t which, const void* d_plane) {
    if (!e || (which != 0 && which != 1)) return VC_ERR_ARG;
    if (bind_device(e)) return VC_ERR_CUDA;
    bool& valid = which == 0 ? e->halo_lo : e->halo_hi;
    if (!d_plane) { valid = false; return VC_OK; }
    int rc = ensure_volumes(e);
    if (rc) return rc;
    uint32_t* dst = halo_slot(e, which);
    if (!dst) return fail(e, VC_ERR_ARG, "vc_import_halo: plane %s of slab [%d,%d) lies outside the grid (it is empty by definition, Model.h:119-124)",
                          which == 0 ? "z_begin - 1" : "z_end", e->g.z_begin, e->g.z_end);
    vol_grant_access(d_plane, e->g.device);  // a neighbour engine's plane in this process (vc_export_halo) may live in memory not yet mapped here
    VC_CUDA(e, cudaMemcpyAsync(dst, d_plane, (size_t)e->plane_words * 4, cudaMemcpyDefault, e->stream));
    valid = true;
    e->have_colors = false;
    e->have_mc = false;
    return VC_OK;
}

int vc_exchange_halos_peer(vc_engine** engines, int32_t n) {
    if (!engines || n < 1) return VC_ERR_ARG;
    std::vector<vc_engine*> es(engines, engines + n);
    for (vc_engine* e : es) if (!e) return VC_ERR_ARG;
    std::sort(es.begin(), es.end(), [](const vc_engine* a, const vc_engine* b) { return a->g.z_begin < b->g.z_begin; });
    vc_engine* e0 = es[0];
    for (int i = 0; i < n; i++) {
        vc_engine* e = es[i];
        if (e->g.X != e0->g.X || e->g.Y != e0->g.Y || e->g.Z != e0->g.Z) return fail(e, VC_ERR_ARG, "vc_exchange_halos_peer: engines of different grids");
        if (i + 1 < n && e->g.z_end != es[i + 1]->g.z_begin)
            return fail(e, VC_ERR_ARG, "vc_exchange_halos_peer: slabs [%d,%d) and [%d,%d) are not adjacent", e->g.z_begin, e->g.z_end, es[i + 1]->g.z_begin, es[i + 1]->g.z_end);
        if (bind_device(e)) return VC_ERR_CUDA;
        int rc = materialize_reset(e);
        if (rc) return rc;
        if (!e->ev_halo) VC_CUDA(e, cudaEventCreateWithFlags(&e->ev_halo, cudaEventDisableTiming));
        VC_CUDA(e, cudaEventRecord(e->ev_halo, e->stream));  // my slab is complete here
    }
    const size_t bytes = (size_t)e0->plane_words * 4;
    for (int i = 0; i + 1 < n; i++) {
        vc_engine *a = es[i], *b = es[i + 1];  // a below b: a's last plane is b's z_begin - 1, b's first plane is a's z_end
        grant_peer_access(a, b->g.device); grant_peer_access(b, a->g.device);
        if (bind_device(b)) return VC_ERR_CUDA;
        VC_CUDA(b, cudaStreamWaitEvent(b->stream, a->ev_halo, 0));
        VC_CUDA(b, cudaMemcpyAsync(halo_slot(b, 0), a->occ_slab() + a->slab_words - a->plane_words, bytes, cudaMemcpyDefault, b->stream));
        b->halo_lo = true; b->have_colors = false; b->have_mc = false;
        if (bind_device(a)) return VC_ERR_CUDA;
        VC_CUDA(a, cudaStreamWaitEvent(a->stream, b->ev_halo, 0));
        VC_CUDA(a, cudaMemcpyAsync(halo_slot(a, 1), b->occ_slab(), bytes, cudaMemcpyDefault, a->stream));
        a->halo_hi = true; a->have_colors = false; a->have_mc = false;
    }
    return VC_OK;
}

int vc_gather_peer(vc_engine** engines, int32_t n, int32_t what) {
    if (!engines || n < 1 || !(what & 3) || (what & ~3)) return VC_ERR_ARG;
    std::vector<vc_engine*> es(engines, engines + n);
    for (vc_engine* e : es) if (!e) return VC_ERR_ARG;
    std::sort(es.begin(), es.end(), [](const vc_engine* a, const vc_engine* b) { return a->g.z_begin < b->g.z_begin; });
    vc_engine* e0 = es[0];
    if (e0->g.z_begin != 0 || es[n - 1]->g.z_end != e0->g.Z) return fail(e0, VC_ERR_ARG, "vc_gather_peer: the slabs do not cover [0,%d)", e0->g.Z);
    for (int i = 0; i < n; i++) {
        vc_engine* e = es[i];
        if (e->g.X != e0->g.X || e->g.Y != e0->g.Y || e->g.Z != e0->g.Z) return fail(e, VC_ERR_ARG, "vc_gather_peer: engines of different grids");
        if (i + 1 < n && e->g.z_end != es[i + 1]->g.z_begin) return fail(e, VC_ERR_ARG, "vc_gather_peer: slabs [%d,%d) and [%d,%d) are not adjacent", e->g.z_begin, e->g.z_end, es[i + 1]->g.z_begin, es[i + 1]->g.z_end);
        if (!e->d_occ_full) return fail(e, VC_ERR_STATE, "vc_gather_peer: every engine needs whole-grid buffers (vc_alloc_full_volumes / vc_bind_volumes)");
        if (bind_device(e)) return VC_ERR_CUDA;
        int rc = materialize_reset(e);
        if (rc) return rc;
        for (int k = 0; k < n; k++) {  // direct loads / stores over NVLink instead of staging through the host
            if (es[k]->g.device == e->g.device) continue;
            grant_peer_access(e, es[k]->g.device);
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, e->g.device, es[k]->g.device) == cudaSuccess && can) {
                const cudaError_t pe = cudaDeviceEnablePeerAccess(es[k]->g.device, 0);
                if (pe != cudaSuccess) cudaGetLastError();  // already enabled
            }
        }
        if (!e->ev_halo) VC_CUDA(e, cudaEventCreateWithFlags(&e->ev_halo, cudaEventDisableTiming));
        VC_CUDA(e, cudaEventRecord(e->ev_halo, e->stream));  // my slab is complete here
    }
    const size_t pw = (size_t)e0->plane_words;
    for (int d = 0; d < n; d++) {  // every engine pulls the other slabs on its own stream, starting with its upper neighbour
        vc_engine* dst = es[d];
        if (bind_device(dst)) return VC_ERR_CUDA;
        for (int k = 1; k < n; k++) {
            vc_engine* src = es[(d + k) % n];
            const size_t off = (size_t)src->g.z_begin * pw, bytes = (size_t)src->slab_words * 4;
            VC_CUDA(dst, cudaStreamWaitEvent(dst->stream, src->ev_halo, 0));
            if (what & 1) VC_CUDA(dst, cudaMemcpyPeerAsync(dst->d_occ_full + off, dst->g.device, src->d_occ_full + off, src->g.device, bytes, dst->stream));
            if (what & 2) VC_CUDA(dst, cudaMemcpyPeerAsync(dst->d_seen_full + off, dst->g.device, src->d_seen_full + off, src->g.device, bytes, dst->stream));
        }
        if (what & 1) { dst->gathered = true; dst->have_colors = false; dst->have_mc = false; }
    }
    return VC_OK;
}

int vc_comm_unique_id(void* unique_id_128) {
    if (!unique_id_128) return VC_ERR_ARG;
    const NcclApi* api = load_nccl();
    if (!api) return fail(nullptr, VC_ERR_COMM, "vc_comm_unique_id: %s", g_nccl.error.c_str());
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    ncclResult_t r = api->GetUniqueId(&id);
    if (r != ncclSuccess) return fail(nullptr, VC_ERR_COMM, "ncclGetUniqueId failed: %s", api->GetErrorString(r));
    memcpy(unique_id_128, &id, sizeof id);
    return VC_OK;
}

int vc_comm_init(vc_engine* e, int32_t rank, int32_t world, const void* unique_id_128) {
    if (!e) return VC_ERR_ARG;
    if (!unique_id_128 || world < 1 || rank < 0 || rank >= world) return fail(e, VC_ERR_ARG, "vc_comm_init: bad rank %d / world %d / id", rank, world);
    if (e->comm) return fail(e, VC_ERR_STATE, "vc_comm_init: communicator already initialised (vc_comm_destroy first)");
    const NcclApi* api = load_nccl();
    if (!api) return fail(e, VC_ERR_COMM, "vc_comm_init: %s", g_nccl.error.c_str());
    if (bind_device(e)) return VC_ERR_CUDA;
    ncclUniqueId id;
    memcpy(&id, unique_id_128, sizeof id);
    VC_NCCL(e, api, api->CommInitRank(&e->comm, world, id, rank));  // blocks until every rank has called it
    e->comm_rank = rank;
    e->comm_world = world;
    return VC_OK;
}

int vc_comm_destroy(vc_engine* e) {
    if (!e) return VC_ERR_ARG;
    if (!e->comm) return VC_OK;
    const NcclApi* api = load_nccl();
    cudaSetDevice(e->g.device);
    cudaStreamSynchronize(e->stream);
    if (api) api->CommDestroy(e->comm);
    e->comm = nullptr;
    e->comm_rank = 0; e->comm_world = 1;
    return VC_OK;
}

int vc_comm_info(const vc_engine* e, int32_t* rank, int32_t* world, int32_t* nccl_version) {
    if (!e || !rank || !world || !nccl_version) return VC_ERR_ARG;
    *rank = e->comm ? e->comm_rank : 0;
    *world = e->comm ? e->comm_world : 1;
    *nccl_version = e->comm ? g_nccl.version : 0;
    return VC_OK;
}

int vc_exchange_halos(vc_engine* e) {
    if (!e) return VC_ERR_ARG;
    if (!e->comm) return fail(e, VC_ERR_STATE, "vc_exchange_halos: no communicator (vc_comm_init)");
    const NcclApi* api = load_nccl();
    if (bind_device(e)) return VC_ERR_CUDA;
    int rc = materialize_reset(e);
    if (rc) return rc;
    // slabs are in rank order along z (rank r below rank r + 1): my first plane goes down, my last plane goes up
    const bool down = e->comm_rank > 0 && e->g.z_begin > 0, up = e->comm_rank + 1 < e->comm_world && e->g.z_end < e->g.Z;
    const size_t n = (size_t)e->plane_words;
    VC_NCCL(e, api, api->GroupStart());
    if (down) {
        VC_NCCL(e, api, api->Send(e->occ_slab(), n, ncclUint32, e->comm_rank - 1, e->comm, e->stream));
        VC_NCCL(e, api, api->Recv(halo_slot(e, 0), n, ncclUint32, e->comm_rank - 1, e->comm, e->stream));
    }
    if (up) {
        VC_NCCL(e, api, api->Send(e->occ_slab() + e->slab_words - e->plane_words, n, ncclUint32, e->comm_rank + 1, e->comm, e->stream));
        VC_NCCL(e, api, api->Recv(halo_slot(e, 1), n, ncclUint32, e->comm_rank + 1, e->comm, e->stream));
    }
    VC_NCCL(e, api, api->GroupEnd());
    if (down) e->halo_lo = true;
    if (up) e->halo_hi = true;
    e->have_colors = false;
    e->have_mc = false;
    return VC_OK;
}

int vc_gather(vc_engine* e, int32_t what, const int32_t* z_bounds) {
    if (!e) return VC_ERR_ARG;
    if (!e->comm) return fail(e, VC_ERR_STATE, "vc_gather: no communicator (vc_comm_init)");
    if (!(what & 3) || (what & ~3) || !z_bounds) return fail(e, VC_ERR_ARG, "vc_gather: what = 1 (occupied), 2 (seen) or 3 (both), with the world + 1 slab boundaries");
    if (!e->d_occ_full) return fail(e, VC_ERR_STATE, "vc_gather: needs whole-grid buffers (vc_alloc_full_volumes or vc_bind_volumes)");
    const int R = e->comm_world, r = e->comm_rank;
    if (z_bounds[0] != 0 || z_bounds[R] != e->g.Z || z_bounds[r] != e->g.z_begin || z_bounds[r + 1] != e->g.z_end)
        return fail(e, VC_ERR_ARG, "vc_gather: z_bounds do not cover [0,%d) with slab %d = [%d,%d)", e->g.Z, r, e->g.z_begin, e->g.z_end);
    bool equal = true;
    for (int k = 0; k < R; k++) {
        if (z_bounds[k + 1] <= z_bounds[k]) return fail(e, VC_ERR_ARG, "vc_gather: empty slab %d", k);
        equal = equal && (z_bounds[k + 1] - z_bounds[k] == z_bounds[1] - z_bounds[0]);
    }
    const NcclApi* api = load_nccl();
    if (bind_device(e)) return VC_ERR_CUDA;
    int rc = materialize_reset(e);
    if (rc) return rc;
    const size_t pw = (size_t)e->plane_words;
    for (int vol = 0; vol < 2; vol++) {
        if (!(what & (1 << vol))) continue;
        uint32_t* full = vol == 0 ? e->d_occ_full : e->d_seen_full;
        if (equal) {  // in place: my slab already sits at rank * count
            VC_NCCL(e, api, api->AllGather(full + (size_t)z_bounds[r] * pw, full, (size_t)(z_bounds[1] - z_bounds[0]) * pw, ncclUint32, e->comm, e->stream));
        } else {      // ragged (balanced) slabs: every rank sends its slab to every other one, all transfers in one group
            VC_NCCL(e, api, api->GroupStart());
            for (int k = 0; k < R; k++) {
                if (k == r) continue;
                VC_NCCL(e, api, api->Send(full + (size_t)z_bounds[r] * pw, (size_t)(z_bounds[r + 1] - z_bounds[r]) * pw, ncclUint32, k, e->comm, e->stream));
                VC_NCCL(e, api, api->Recv(full + (size_t)z_bounds[k] * pw, (size_t)(z_bounds[k + 1] - z_bounds[k]) * pw, ncclUint32, k, e->comm, e->stream));
            }
            VC_NCCL(e, api, api->GroupEnd());
        }
    }
    if (what & 1) { e->gathered = true; e->have_colors = false; e->have_mc = false; }
    return VC_OK;
}

int vc_download_full(vc_engine* e, int32_t which, uint32_t* words, uint64_t n_words) {
    if (!e || !words || (which != 0 && which != 1)) return VC_ERR_ARG;
    if (!e->d_occ_full) return fail(e, VC_ERR_STATE, "vc_download_full: no whole-grid buffers (vc_alloc_full_volumes / vc_bind_volumes)");
    if (which == 0 && !e->gathered && !e->whole_grid()) return fail(e, VC_ERR_STATE, "vc_download_full: the grid has not been gathered (vc_gather / vc_set_gathered)");
    const uint64_t n = (uint64_t)e->g.Z * (uint64_t)e->plane_words;
    if (n_words < n) return fail(e, VC_ERR_CAPACITY, "vc_download_full: buffer holds %llu words, the grid has %llu", (unsigned long long)n_words, (unsigned long long)n);
    if (bind_device(e)) return VC_ERR_CUDA;
    int rc = materialize_reset(e);
    if (rc) return rc;
    VC_CUDA(e, cudaMemcpyAsync(words, which == 0 ? e->d_occ_full : e->d_seen_full, n * 4, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

int vc_comm_allreduce_u64(vc_engine* e, uint64_t* values, int32_t n) {
    if (!e || !values || n < 1) return VC_ERR_ARG;
    if (!e->comm) return VC_OK;  // a single engine: the sum is the value
    const NcclApi* api = load_nccl();
    if (bind_device(e)) return VC_ERR_CUDA;
    if (e->reduce_cap < (size_t)n) {
        VC_CUDA(e, cudaStreamSynchronize(e->stream));
        cudaFree(e->d_reduce); e->d_reduce = nullptr; e->reduce_cap = 0;
        VC_CUDA(e, cudaMalloc(&e->d_reduce, (size_t)n * 8));
        e->reduce_cap = (size_t)n;
    }
    VC_CUDA(e, cudaMemcpyAsync(e->d_reduce, values, (size_t)n * 8, cudaMemcpyHostToDevice, e->stream));
    VC_NCCL(e, api, api->AllReduce(e->d_reduce, e->d_reduce, (size_t)n, ncclUint64, ncclSum, e->comm, e->stream));
    VC_CUDA(e, cudaMemcpyAsync(values, e->d_reduce, (size_t)n * 8, cudaMemcpyDeviceToHost, e->stream));
    VC_CUDA(e, cudaStreamSynchronize(e->stream));
    return VC_OK;
}

}  // extern "C"
