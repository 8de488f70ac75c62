/*
 * voxcarve_oracle.c — CPU restatement of the reference voxel hot path.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT. Only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py may load this. The product
 * (libvoxcarve.so) never links, imports or calls anything in oracle/.
 *
 * Parity pin: the projection arithmetic below is checked bit-for-bit against
 * cv2.gemm 4.13.0 (tests/golden/gemm_kat.npz, 52 800 vectors incl. adversarial
 * near-tie rows) and the whole carve/colour loop against a literal per-voxel
 * cv2.gemm run of the reference algorithm (tests/golden/{box,human}_literal.npz);
 * generator: tools/make_goldens.py. The reference C++ itself cannot be built here
 * (needs OpenCV C++ + Eigen, neither installed) so there is no oracle/_ref.
 * Not pinned by any reference fixture (recalled from OpenCV matx.hpp): the f64
 * accumulation inside cv::norm(Vec4f) used for the colour depth (vo_depth).
 *
 * Every function cites the reference lines it restates (paths under /root/reference/src).
 * Build: make -C oracle   (gcc -O2 -ffp-contract=off -pthread)
 */
#include <math.h>
#include <stdio.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <stdatomic.h>
#include <unistd.h>

#define VO_API __attribute__((visibility("default")))

/* VoxelCarving.cpp:19 first product `intr * pose` (3x3 . 3x4, CV_32F): OpenCV's small
 * matrix path = plain f32, left to right, no FMA [pinned: gemm_kat.npz KM]. */
VO_API void vo_gemm3x3_3x4(const float* K, const float* M, float* P) {
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 4; j++) {
            float a = K[i * 3 + 0] * M[0 * 4 + j]; /* -ffp-contract=off: no FMA */
            float b = K[i * 3 + 1] * M[1 * 4 + j];
            float c = K[i * 3 + 2] * M[2 * 4 + j];
            float t = a + b;
            P[i * 4 + j] = t + c;
        }
}

/* VoxelCarving.cpp:19 second product `(intr*pose) * world` (3x4 . 4x1, CV_32F):
 * products and a SEQUENTIAL accumulation ((s0+s1)+s2)+s3 in f64, one rounding to f32
 * [pinned: gemm_kat.npz proj; SURVEY §8c-5 states a different association, which the
 * near-tie vectors refute]. */
VO_API void vo_project(const float* P, const float* w, float* proj) {
    for (int i = 0; i < 3; i++) {
        double s = (double)P[i * 4 + 0] * (double)w[0];
        s = s + (double)P[i * 4 + 1] * (double)w[1];
        s = s + (double)P[i * 4 + 2] * (double)w[2];
        s = s + (double)P[i * 4 + 3] * (double)w[3];
        proj[i] = (float)s;
    }
}

/* Model.h:134-136 toWord: (y*size, x*size, -1*z*size, 1) — int*float products in f32. */
VO_API void vo_world(int x, int y, int z, float s, float* w) {
    w[0] = (float)y * s;
    w[1] = (float)x * s;
    w[2] = (float)(-1 * z) * s;
    w[3] = 1.0f;
}

/* VoxelCarving.cpp:44 `(int)std::round(float)`: half away from zero; NaN, inf and
 * values outside int range convert to INT_MIN on x86 (cvttss2si), i.e. out of bounds. */
VO_API int32_t vo_round_to_int(float v) {
    float r = roundf(v);
    if (!(r >= -2147483648.0f && r < 2147483648.0f)) return INT32_MIN;
    return (int32_t)r;
}

/* VoxelCarving.cpp:18-21 + :44: pixel of a voxel in one view. Returns 1 if inside the image (:45). */
static inline int vo_pixel(const float* P, int x, int y, int z, float s, int W, int H, int* px, int* py) {
    float w[4], p[3];
    vo_world(x, y, z, s, w);
    vo_project(P, w, p);
    float u = p[0] / p[2], v = p[1] / p[2]; /* :20, IEEE f32 divides, no depth-sign test */
    *px = vo_round_to_int(u);
    *py = vo_round_to_int(v);
    return *px >= 0 && *px < W && *py >= 0 && *py < H; /* cv::Point::inside(Rect(0,0,W,H)) */
}

VO_API int vo_pixel_of(const float* P, int x, int y, int z, float s, int W, int H, int* px, int* py, float* uv) {
    float w[4], p[3];
    vo_world(x, y, z, s, w);
    vo_project(P, w, p);
    uv[0] = p[0] / p[2];
    uv[1] = p[1] / p[2];
    return vo_pixel(P, x, y, z, s, W, H, px, py);
}

static inline int mask_is_bg(const uint32_t* bits, const uint8_t* bgr, int v, int W, int H, int px, int py) {
    if (bits) {
        int Ww = (W + 31) / 32;
        return (bits[((size_t)v * H + py) * Ww + (px >> 5)] >> (px & 31)) & 1u;
    }
    const uint8_t* p = bgr + (((size_t)v * H + py) * W + px) * 3;
    return p[0] == 0 && p[1] == 0 && p[2] == 0; /* VoxelCarving.cpp:50 */
}

/* One z-range of VoxelCarving.cpp:60-72 (views outer) / :39-55 (x, y, z loops in the order
 * of Model.h:10-35), on byte-per-voxel scratch indexed like Model::flatten (Model.h:104-106). */
static void carve_range(int X, int Y, int zlo, int zhi, int z0, float s, int V, int W, int H, const float* P,
                        const uint32_t* bits, const uint8_t* bgr, uint8_t* occ8, uint8_t* seen8) {
    for (int v = 0; v < V; v++) {
        const float* Pv = P + (size_t)v * 12;
        for (int x = 0; x < X; x++)
            for (int y = 0; y < Y; y++)
                for (int z = zlo; z < zhi; z++) {
                    int px, py;
                    if (!vo_pixel(Pv, x, y, z, s, W, H, &px, &py)) continue; /* :45-48 */
                    size_t f = (size_t)x + (size_t)X * ((size_t)y + (size_t)Y * (size_t)(z - z0));
                    if (mask_is_bg(bits, bgr, v, W, H, px, py)) occ8[f] = 0; /* :50-53 */
                    seen8[f] = 1;                                            /* :54 */
                }
    }
}

static void pack_bits(const uint8_t* b8, int X, int Y, int nz, uint32_t* words) {
    int Wx = (X + 31) / 32;
    for (size_t row = 0; row < (size_t)Y * nz; row++)
        for (int j = 0; j < Wx; j++) {
            uint32_t wd = 0;
            for (int b = 0; b < 32 && j * 32 + b < X; b++) wd |= (uint32_t)(b8[row * X + j * 32 + b] != 0) << b;
            words[row * Wx + j] = wd;
        }
}

typedef struct {
    int X, Y, z0, z1, V, W, H;
    float s;
    const float* P;
    const uint32_t* bits;
    const uint8_t* bgr;
    uint8_t *occ8, *seen8;
    atomic_int next_z;
} carve_job;

static void* carve_worker(void* arg) {
    carve_job* j = (carve_job*)arg;
    for (;;) { /* z-planes are independent (flatten is z-major), so threads take one plane at a time */
        int z = atomic_fetch_add(&j->next_z, 1);
        if (z >= j->z1) break;
        carve_range(j->X, j->Y, z, z + 1, j->z0, j->s, j->V, j->W, j->H, j->P, j->bits, j->bgr, j->occ8, j->seen8);
    }
    return NULL;
}

VO_API int vo_max_threads(void) {
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n < 1 ? 1 : (int)n;
}

/* What the reference computes for every voxel of a box, summarised: [0] every voxel inside the image, [1] none inside,
 * [2..5] min / max of px and of py (INT32_MIN for NaN / out-of-range coordinates, as vo_round_to_int), [6] some voxel has a
 * depth proj_2 <= 0 or not finite. */
typedef struct {
    const float* P;
    float s;
    int W, H, x0, y0, x1, y1, z1;
    atomic_int next_z;
    pthread_mutex_t lock;
    int32_t acc[7];
} bounds_job;

static void bounds_fold(int32_t* acc, const int32_t* b) {
    acc[0] &= b[0]; acc[1] &= b[1]; acc[6] |= b[6];
    for (int k = 2; k < 6; k += 2) {
        if (b[k] < acc[k]) acc[k] = b[k];
        if (b[k + 1] > acc[k + 1]) acc[k + 1] = b[k + 1];
    }
}

static void* bounds_worker(void* arg) {
    bounds_job* j = (bounds_job*)arg;
    int32_t b[7] = {1, 1, INT32_MAX, INT32_MIN, INT32_MAX, INT32_MIN, 0};
    for (;;) {
        int z = atomic_fetch_add(&j->next_z, 1);
        if (z > j->z1) break;
        for (int y = j->y0; y <= j->y1; y++)
            for (int x = j->x0; x <= j->x1; x++) {
                float w[4], p[3];
                int px, py;
                vo_world(x, y, z, j->s, w);
                vo_project(j->P, w, p);
                int in = vo_pixel(j->P, x, y, z, j->s, j->W, j->H, &px, &py);
                b[0] &= in; b[1] &= !in;
                if (!(p[2] > 0.0f) || !isfinite(p[2])) b[6] = 1;
                if (px < b[2]) b[2] = px;
                if (px > b[3]) b[3] = px;
                if (py < b[4]) b[4] = py;
                if (py > b[5]) b[5] = py;
            }
    }
    pthread_mutex_lock(&j->lock);
    bounds_fold(j->acc, b);
    pthread_mutex_unlock(&j->lock);
    return NULL;
}

/* box = voxels [x0, x1] x [y0, y1] x [z0, z1] (inclusive); z-planes split over nthreads pthreads (< 1: all online cores) */
VO_API int vo_box_pixel_bounds(const float* P, float s, int W, int H, int x0, int y0, int z0, int x1, int y1, int z1, int nthreads, int32_t* out) {
    if (x1 < x0 || y1 < y0 || z1 < z0) return -1;
    bounds_job job = {P, s, W, H, x0, y0, x1, y1, z1, 0, PTHREAD_MUTEX_INITIALIZER, {1, 1, INT32_MAX, INT32_MIN, INT32_MAX, INT32_MIN, 0}};
    atomic_store(&job.next_z, z0);
    if (nthreads < 1) nthreads = vo_max_threads();
    if (nthreads > z1 - z0 + 1) nthreads = z1 - z0 + 1;
    if (nthreads == 1) {
        bounds_worker(&job);
    } else {
        pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * nthreads);
        for (int t = 0; t < nthreads; t++) pthread_create(&th[t], NULL, bounds_worker, &job);
        for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
        free(th);
    }
    memcpy(out, job.acc, sizeof job.acc);
    return 0;
}

/* carve() VoxelCarving.cpp:60-72 on the z-slab [z0,z1) of an X*Y*Z grid. Exactly one of
 * mask_bits / mask_bgr is non-NULL. Outputs bit volumes word[((z-z0)*Y + y)*ceil(X/32) + (x>>5)],
 * bit x&31; occupied starts all-ones (Model.cpp:9-14, alpha = 1), seen all-zero.
 * nthreads = 1 is the reference as written (single thread); nthreads > 1 splits z-planes over
 * pthreads (nthreads < 1: all online cores). */
VO_API int vo_carve(int X, int Y, int Z, float s, int z0, int z1, int V, int W, int H, const float* P,
                    const uint32_t* mask_bits, const uint8_t* mask_bgr, uint32_t* occ, uint32_t* seen,
                    int nthreads) {
    if (X < 1 || Y < 1 || Z < 1 || z0 < 0 || z1 > Z || z0 >= z1 || (!mask_bits == !mask_bgr)) return -1;
    int nz = z1 - z0;
    size_t n = (size_t)X * Y * nz;
    uint8_t* occ8 = (uint8_t*)malloc(n);
    uint8_t* seen8 = (uint8_t*)calloc(n, 1);
    if (!occ8 || !seen8) return -2;
    memset(occ8, 1, n);
    if (nthreads < 1) nthreads = vo_max_threads();
    if (nthreads > nz) nthreads = nz;
    carve_job job = {X, Y, z0, z1, V, W, H, s, P, mask_bits, mask_bgr, occ8, seen8, 0};
    atomic_store(&job.next_z, z0);
    if (nthreads == 1) {
        carve_range(X, Y, z0, z1, z0, s, V, W, H, P, mask_bits, mask_bgr, occ8, seen8);
    } else {
        pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * nthreads);
        for (int t = 0; t < nthreads; t++) pthread_create(&th[t], NULL, carve_worker, &job);
        for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
        free(th);
    }
    pack_bits(occ8, X, Y, nz, occ);
    pack_bits(seen8, X, Y, nz, seen);
    free(occ8);
    free(seen8);
    return 0;
}

static inline int getbit(const uint32_t* w, int X, int Y, int Z, int x, int y, int z) {
    if (x < 0 || x >= X || y < 0 || y >= Y || z < 0 || z >= Z) return 0; /* Model::get OOB -> alpha 0 (Model.h:119-124) */
    int Wx = (X + 31) / 32;
    return (w[((size_t)z * Y + y) * Wx + (x >> 5)] >> (x & 31)) & 1u;
}
static inline void putbit(uint32_t* w, int X, int Y, int x, int y, int z, int v) {
    int Wx = (X + 31) / 32;
    uint32_t* p = &w[((size_t)z * Y + y) * Wx + (x >> 5)];
    if (v) *p |= 1u << (x & 31); else *p &= ~(1u << (x & 31));
}

/* fastCarve() VoxelCarving.cpp:74-167: BFS from (0,0,0); `visited` is the seen bit (Model.h:154-160). */
VO_API int vo_fast_carve(int X, int Y, int Z, float s, int V, int W, int H, const float* P,
                         const uint32_t* mask_bits, const uint8_t* mask_bgr, uint32_t* occ, uint32_t* seen) {
    int Wx = (X + 31) / 32;
    size_t nw = (size_t)Wx * Y * Z;
    memset(seen, 0, nw * 4);
    for (size_t i = 0; i < nw; i++) /* Model ctor: every voxel occupied; row padding bits stay 0 */
        occ[i] = ((i % Wx) == (size_t)Wx - 1 && X % 32) ? (1u << (X % 32)) - 1 : 0xffffffffu;
    size_t cap = 1 << 16, head = 0, tail = 0;
    int32_t* q = (int32_t*)malloc(cap * 3 * sizeof(int32_t));
    if (!q) return -2;
#define PUSH(a, b, c) do { if (tail == cap) { cap *= 2; q = (int32_t*)realloc(q, cap * 3 * sizeof(int32_t)); if (!q) return -2; } \
        q[tail * 3] = (a); q[tail * 3 + 1] = (b); q[tail * 3 + 2] = (c); tail++; } while (0)
    PUSH(0, 0, 0); /* :101 */
    while (head < tail) {
        int x = q[head * 3], y = q[head * 3 + 1], z = q[head * 3 + 2];
        head++;
        if (getbit(seen, X, Y, Z, x, y, z)) continue; /* :107 */
        putbit(seen, X, Y, x, y, z, 1);               /* :110 */
        int carved = 0;
        for (int v = 0; v < V; v++) { /* :113-130 */
            int px, py;
            if (!vo_pixel(P + (size_t)v * 12, x, y, z, s, W, H, &px, &py)) continue;
            if (mask_is_bg(mask_bits, mask_bgr, v, W, H, px, py)) { putbit(occ, X, Y, x, y, z, 0); carved = 1; break; }
        }
        if (carved) { /* :132-163 */
            if (x > 0 && !getbit(seen, X, Y, Z, x - 1, y, z)) PUSH(x - 1, y, z);
            if (x < X - 1 && !getbit(seen, X, Y, Z, x + 1, y, z)) PUSH(x + 1, y, z);
            if (y > 0 && !getbit(seen, X, Y, Z, x, y - 1, z)) PUSH(x, y - 1, z);
            if (y < Y - 1 && !getbit(seen, X, Y, Z, x, y + 1, z)) PUSH(x, y + 1, z);
            if (z > 0 && !getbit(seen, X, Y, Z, x, y, z - 1)) PUSH(x, y, z - 1);
            if (z < Z - 1 && !getbit(seen, X, Y, Z, x, y, z + 1)) PUSH(x, y, z + 1);
        }
    }
#undef PUSH
    free(q);
    return 0;
}

/* ColorReconstruction.h:59 depth = cv::norm(cameras[i] - word_coord): Vec4f difference in f32,
 * squares accumulated in f64, sqrt, narrowed to the `float depth` of Model::addColor (Model.h:142). */
VO_API float vo_depth(const float* cam4, const float* w4) {
    double acc = 0;
    for (int k = 0; k < 4; k++) {
        float d = cam4[k] - w4[k];
        acc += (double)d * (double)d;
    }
    return (float)sqrt(acc);
}

/* voxel_pass_loops (ColorReconstruction.h:34-74) + body reconstructClosestColor (.cpp:33-41, mode 1)
 * or reconstructAvgColor (.cpp:59-66, mode 2), on a full-grid occupancy bit volume.
 * Emits one record per SURFACE voxel (alpha != 0 && !isInner, .h:46) in ascending flatten order
 * z,y,x: idx = x + X*(y + Y*z), rgbn = (r, g, b, min(n_observations, 255)); voxels with n = 0 keep
 * MODEL_COLOR (50,168,141) because the body `continue`s (.cpp:29-31). Returns the record count
 * (counts beyond cap are still counted, not written). */
VO_API uint64_t vo_color(int X, int Y, int Z, float s, int V, int W, int H, const float* P, const float* M,
                         const uint8_t* images_bgr, const uint32_t* occ, int mode, uint64_t* idx_out,
                         uint8_t* rgbn_out, uint64_t cap) {
    uint64_t n = 0;
    for (int z = 0; z < Z; z++)
        for (int y = 0; y < Y; y++)
            for (int x = 0; x < X; x++) {
                if (!getbit(occ, X, Y, Z, x, y, z)) continue;
                int inner = getbit(occ, X, Y, Z, x - 1, y, z) && getbit(occ, X, Y, Z, x + 1, y, z) &&
                            getbit(occ, X, Y, Z, x, y - 1, z) && getbit(occ, X, Y, Z, x, y + 1, z) &&
                            getbit(occ, X, Y, Z, x, y, z - 1) && getbit(occ, X, Y, Z, x, y, z + 1); /* Model.h:126-132 */
                if (inner) continue;
                float w[4];
                vo_world(x, y, z, s, w);
                int nobs = 0;
                float sum[3] = {0, 0, 0}, best[3] = {50, 168, 141}, bestd = 0;
                for (int v = 0; v < V; v++) {
                    int px, py;
                    if (!vo_pixel(P + (size_t)v * 12, x, y, z, s, W, H, &px, &py)) continue; /* .h:54-57 */
                    const uint8_t* pix = images_bgr + (((size_t)v * H + py) * W + px) * 3;   /* .h:58 */
                    float rgb[3] = {(float)pix[2], (float)pix[1], (float)pix[0]};            /* .h:59 BGR->RGB */
                    float cam[4] = {M[v * 12 + 3], M[v * 12 + 7], M[v * 12 + 11], 1.0f};     /* .h:21 */
                    float d = vo_depth(cam, w);
                    if (nobs == 0 || d < bestd) { bestd = d; memcpy(best, rgb, sizeof best); } /* .cpp:34-40 */
                    for (int c = 0; c < 3; c++) sum[c] = sum[c] + rgb[c];                     /* .cpp:60-64 */
                    nobs++;
                }
                uint8_t out[4] = {50, 168, 141, (uint8_t)(nobs > 255 ? 255 : nobs)}; /* MODEL_COLOR, Model.h:90 */
                if (nobs > 0) {
                    for (int c = 0; c < 3; c++) {
                        float val = mode == 2 ? roundf(sum[c] / (float)nobs) : best[c]; /* .cpp:65-66 */
                        out[c] = (uint8_t)val;
                    }
                }
                if (n < cap) {
                    idx_out[n] = (uint64_t)x + (uint64_t)X * ((uint64_t)y + (uint64_t)Y * (uint64_t)z);
                    memcpy(rgbn_out + n * 4, out, 4);
                }
                n++;
            }
    return n;
}

/* number of triangles of each of the 256 cube configurations = entries of triTable[idx] / 3
 * (MarchingCubes.h:147-404); filled by the caller from the shared table file so that oracle and
 * product do not share code — see oracle/oracle.py. */
VO_API void vo_mc_classify(int X, int Y, int Z, const uint32_t* occ, const uint8_t* tri_count256,
                           uint64_t* hist256, uint64_t* n_active, uint64_t* n_tris) {
    memset(hist256, 0, 256 * sizeof(uint64_t));
    *n_active = 0;
    *n_tris = 0;
    for (int x = -1; x < X; x++) /* MarchingCubes.cpp:12-14 */
        for (int y = -1; y < Y; y++)
            for (int z = -1; z < Z; z++) {
                /* corner order MarchingCubes.h:537-552; bit i set iff corner EMPTY (w < 0.5, :479-484) */
                int c[8] = {getbit(occ, X, Y, Z, x + 1, y, z),     getbit(occ, X, Y, Z, x, y, z),
                            getbit(occ, X, Y, Z, x, y + 1, z),     getbit(occ, X, Y, Z, x + 1, y + 1, z),
                            getbit(occ, X, Y, Z, x + 1, y, z + 1), getbit(occ, X, Y, Z, x, y, z + 1),
                            getbit(occ, X, Y, Z, x, y + 1, z + 1), getbit(occ, X, Y, Z, x + 1, y + 1, z + 1)};
                int idx = 0;
                for (int i = 0; i < 8; i++) if (!c[i]) idx |= 1 << i;
                hist256[idx]++;
                if (idx != 0 && idx != 255) (*n_active)++; /* edgeTable[idx] != 0 (:486) */
                *n_tris += tri_count256[idx];
            }
}

/* ------------------------------------------------------------------------------------------------
 * "Next" rows of the hot path (SURVEY §8f): applyClosure and the full marchingCubes on the dense
 * RGBA Model (std::vector<Vector4f> voxels, index = Model::flatten = x + X*(y + Y*z), Model.h:104-106).
 * ---------------------------------------------------------------------------------------------- */
static inline const float* vget(const float* rgba, int X, int Y, int Z, int x, int y, int z) {
    static const float zero[4] = {0, 0, 0, 0}; /* Model::get out of range (Model.h:119-122) */
    if (x < 0 || x >= X || y < 0 || y >= Y || z < 0 || z >= Z) return zero;
    return rgba + 4 * ((size_t)x + (size_t)X * ((size_t)y + (size_t)Y * (size_t)z));
}

/* applyClosure(model, kernelSize) Postprocessing3d.cpp:4-100.  "Dilution" (:20-58): a voxel with w > 0 is kept,
 * any other becomes the mean (sum / count, f32, neighbours visited x, y, z = outer..inner) of its in-grid
 * neighbours with w > 0, or (0,0,0,0).  The erosion (:60-96) tests `w < thresh` with thresh = 0 and can never
 * fire, so the model becomes the dilated copy.  Returns -1 for an even kernel size (:8-11). */
VO_API int vo_closure(int X, int Y, int Z, int kernelSize, const float* in, float* out) {
    if (kernelSize % 2 != 1) return -1;
    const int size = (kernelSize - 1) / 2;
    for (int x = 0; x < X; x++)
        for (int y = 0; y < Y; y++)
            for (int z = 0; z < Z; z++) {
                const float* o = vget(in, X, Y, Z, x, y, z);
                float* dst = out + 4 * ((size_t)x + (size_t)X * ((size_t)y + (size_t)Y * (size_t)z));
                if (o[3] > 0.0f) { memcpy(dst, o, 16); continue; }
                int count = 0;
                float sum[4] = {0, 0, 0, 0};
                for (int i = -size; i <= size; i++) {
                    int xn = x + i;
                    if (xn < 0 || xn >= X) continue;
                    for (int j = -size; j <= size; j++) {
                        int yn = y + j;
                        if (yn < 0 || yn >= Y) continue;
                        for (int k = -size; k <= size; k++) {
                            int zn = z + k;
                            if (zn < 0 || zn >= Z) continue;
                            const float* v = vget(in, X, Y, Z, xn, yn, zn);
                            if (v[3] > 0.0f) { count++; for (int c = 0; c < 4; c++) sum[c] = sum[c] + v[c]; }
                        }
                    }
                }
                if (count > 0) for (int c = 0; c < 4; c++) sum[c] = sum[c] / (float)count;
                memcpy(dst, sum, 16);
            }
    return 0;
}

static int is_default_color(const float* c) { /* MODEL_COLOR / UNSEEN_COLOR heads (Model.h:90-91, MarchingCubes.h:453,457) */
    return (c[0] == 50.0f && c[1] == 168.0f && c[2] == 141.0f) || (c[0] == 204.0f && c[1] == 0.0f && c[2] == 0.0f);
}

/* VertexInterp MarchingCubes.h:428-468 */
static void vertex_interp(float thr, const float* p0, const float* v0, const float* p1, const float* v1, float* coord, float* color) {
    if (v0[3] == 0.0f && v1[3] != 0.0f) { memcpy(color, v1, 12); memcpy(coord, p1, 12); return; }
    if (v0[3] != 0.0f && v1[3] == 0.0f) { memcpy(color, v0, 12); memcpy(coord, p0, 12); return; }
    float f = (v0[3] == v1[3]) ? 0.5f : (thr - v0[3]) / (v1[3] - v0[3]);
    for (int c = 0; c < 3; c++) coord[c] = (1 - f) * p0[c] + f * p1[c];
    if (is_default_color(v0)) memcpy(color, v1, 12);
    else if (is_default_color(v1)) memcpy(color, v0, 12);
    else for (int c = 0; c < 3; c++) color[c] = (1 - f) * v0[c] + f * v1[c];
}

/* marchingCubes() MarchingCubes.cpp:8-31 -> ProcessVoxel MarchingCubes.h:532-578 -> Polygonise :478-511.
 * tri_table = triTable (256 x 16, -1 terminated, MarchingCubes.h:147-404); edgeTable follows from the topology.
 * Output per triangle, in the reference's emission order (x outer, y, z inner): 9 floats (3 unshared vertices, :561-568)
 * and 3 colours MeanColorFloats (:414-416, :570-573, incl. the col[2] = vertex i+1 quirk :506). Returns #triangles. */
VO_API uint64_t vo_marching_cubes(int X, int Y, int Z, const float* rgba, float thr, const int8_t* tri_table, float* verts,
                                  uint32_t* rgb, uint64_t cap) {
    static const int second[12] = {1, 2, 3, 0, 5, 6, 7, 4, 4, 5, 6, 7};
    uint64_t n = 0;
    for (int x = -1; x < X; x++)
        for (int y = -1; y < Y; y++)
            for (int z = -1; z < Z; z++) {
                const int cx[8] = {x + 1, x, x, x + 1, x + 1, x, x, x + 1}, cy[8] = {y, y, y + 1, y + 1, y, y, y + 1, y + 1},
                          cz[8] = {z, z, z, z, z + 1, z + 1, z + 1, z + 1};
                const float* val[8];
                float p[8][3];
                int idx = 0;
                for (int i = 0; i < 8; i++) {
                    val[i] = vget(rgba, X, Y, Z, cx[i], cy[i], cz[i]);
                    p[i][0] = (float)cx[i]; p[i][1] = (float)cy[i]; p[i][2] = (float)cz[i];
                    if (val[i][3] < thr) idx |= 1 << i;
                }
                int edges = 0;
                for (int e = 0; e < 12; e++) if (((idx >> (e % 8)) & 1) != ((idx >> second[e]) & 1)) edges |= 1 << e;
                if (edges == 0) continue;
                float vc[12][3], vcol[12][3];
                for (int e = 0; e < 12; e++)
                    if (edges & (1 << e)) vertex_interp(thr, p[e % 8], val[e % 8], p[second[e]], val[second[e]], vc[e], vcol[e]);
                const int8_t* t = tri_table + idx * 16;
                for (int i = 0; t[i] != -1; i += 3) {
                    if (n < cap) {
                        for (int k = 0; k < 3; k++) memcpy(verts + n * 9 + k * 3, vc[t[i + k]], 12);
                        const float *c0 = vcol[t[i]], *c1 = vcol[t[i + 1]], *c2 = vcol[t[i + 1]];
                        for (int c = 0; c < 3; c++) rgb[n * 3 + c] = (uint32_t)roundf(((c0[c] + c1[c]) + c2[c]) / 3);
                    }
                    n++;
                }
            }
    return n;
}

/* SimpleMesh::WriteMesh MarchingCubes.h:59-87: text .off, ostream default float formatting (== printf %g). */
VO_API int vo_write_off(const char* path, uint64_t ntris, const float* verts, const uint32_t* rgb, float scale, float tx, float ty, float tz) {
    FILE* f = fopen(path, "w");
    if (!f) return -1;
    fprintf(f, "OFF\n%llu %llu 0\n", (unsigned long long)(ntris * 3), (unsigned long long)ntris);
    for (uint64_t i = 0; i < ntris * 3; i++) {
        float a = verts[i * 3] * scale, b = verts[i * 3 + 1] * scale, c = verts[i * 3 + 2] * scale;
        a = a + tx; b = b + ty; c = c + tz;
        fprintf(f, "%g %g %g\n", a, b, c);
    }
    for (uint64_t i = 0; i < ntris; i++)
        fprintf(f, "3 %llu %llu %llu %u %u %u\n", (unsigned long long)(3 * i), (unsigned long long)(3 * i + 1), (unsigned long long)(3 * i + 2),
                rgb[i * 3], rgb[i * 3 + 1], rgb[i * 3 + 2]);
    fclose(f);
    return 0;
}

/* ------------------------------------------------------------------------------------------------
 * cv::undistort as the reference calls it (VoxelCarving.cpp:36,86,89; ColorReconstruction.h:23,26): 8UC3 image,
 * camera matrix K (3x3 f64), distortion (k1 k2 p1 p2 [k3 [k4 k5 k6]]).  The algorithm lives in OpenCV (un-vendored,
 * un-pinned by the reference).  Pinned here to what cv2 4.13.0 computes on x86-64 with its AVX2 code path
 * (tests/golden/undistort_kat.npz, tests/golden/undistort_hostile_kat.npz), W and H below 32767 (remap's limit):
 *   stripes of min(max(1, 4096/W), H) rows; per stripe the new camera matrix K' is K with cy - y0, and the map is
 *   initUndistortRectifyMap(K, dist, I, K', CV_16SC2) in f64:
 *   - ir = K'^-1 by cv::invert's closed form for 3x3 (adjugate times 1/det; all zeros when det == 0);
 *   - row i of the stripe starts at (_x, _y, _w) = fma(i, ir[1|4|7], ir[2|5|8]);
 *   - body, columns [0, W - W%8): blocks of 8 (two AVX2 vectors); the block start advances by 8 ir[0|3|6] per block and
 *     lane l adds l ir[0|3|6]; the polynomials are FMA chains (undistort_body);
 *   - tail, the last W%8 columns: the scalar loop, continuing from the last block start with += ir[0|3|6] per column,
 *     with the FMA contractions the AVX2 build gives it (undistort_tail);
 *   - the thin-prism and tilt stages are identities here, but they turn non-finite intermediates into NaN;
 *   - fixed point: iu = cvRound(u * 32) (round half to even; INT_MIN when NaN or outside int32), sx = iu >> 5,
 *     fx = iu & 31 (same for v); the body saturates sx, sy to int16, the tail wraps them (a (short) cast);
 *   remap INTER_LINEAR, BORDER_CONSTANT(0) with those int16 coordinates: out = (sum_taps src * w + 2^14) >> 15,
 *   w = (32-fx|fx)(32-fy|fy) * 32, taps outside the image read 0.
 * ---------------------------------------------------------------------------------------------- */
static void inv3x3_cv(const double* S, double* t) {  /* cv::invert(DECOMP_LU) for a 3x3 f64 matrix */
#define S_(i, j) S[(i) * 3 + (j)]
    double d = S_(0, 0) * (S_(1, 1) * S_(2, 2) - S_(1, 2) * S_(2, 1)) - S_(0, 1) * (S_(1, 0) * S_(2, 2) - S_(1, 2) * S_(2, 0)) +
               S_(0, 2) * (S_(1, 0) * S_(2, 1) - S_(1, 1) * S_(2, 0));
    if (d == 0) { for (int i = 0; i < 9; i++) t[i] = 0; return; }
    d = 1. / d;
    t[0] = (S_(1, 1) * S_(2, 2) - S_(1, 2) * S_(2, 1)) * d; t[1] = (S_(0, 2) * S_(2, 1) - S_(0, 1) * S_(2, 2)) * d;
    t[2] = (S_(0, 1) * S_(1, 2) - S_(0, 2) * S_(1, 1)) * d; t[3] = (S_(1, 2) * S_(2, 0) - S_(1, 0) * S_(2, 2)) * d;
    t[4] = (S_(0, 0) * S_(2, 2) - S_(0, 2) * S_(2, 0)) * d; t[5] = (S_(0, 2) * S_(1, 0) - S_(0, 0) * S_(1, 2)) * d;
    t[6] = (S_(1, 0) * S_(2, 1) - S_(1, 1) * S_(2, 0)) * d; t[7] = (S_(0, 1) * S_(2, 0) - S_(0, 0) * S_(2, 1)) * d;
    t[8] = (S_(0, 0) * S_(1, 1) - S_(0, 1) * S_(1, 0)) * d;
#undef S_
}
static int cv_round(double v) { /* cvtsd2si / cvtpd2dq: round half to even, INT_MIN when NaN or outside int32 */
    const double r = nearbyint(v);
    return r >= -2147483648.0 && r < 2147483648.0 ? (int)r : INT32_MIN;
}
static double cv_kr(const double* k, double r2) {
    return fma(fma(fma(k[4], r2, k[1]), r2, k[0]), r2, 1.0) / fma(fma(fma(k[7], r2, k[6]), r2, k[5]), r2, 1.0);
}
/* one vector lane: (X, Y, Wh) = block start + lane * ir[0|3|6] */
static void undistort_body(const double* k, double fx, double fy, double u0, double v0, double X, double Y, double Wh, double* u, double* v) {
    const double m = 1.0 / Wh, x = X * m, y = Y * m;
    const double xx = x * x, yy = y * y, r2 = xx + yy, kr = cv_kr(k, r2);
    const double xy2 = (x * y) * 2.0;
    double xd = fma(fma(2.0, xx, r2), k[3], x * kr), yd = fma(fma(2.0, yy, r2), k[2], y * kr);
    xd = fma(k[2], xy2, xd); yd = fma(k[3], xy2, yd);
    const double r4 = r2 * r2;
    const int finite = isfinite(r4) && isfinite(xd) && isfinite(yd);  /* else the thin-prism / tilt terms give NaN */
    *u = finite ? fma(fx, xd, u0) : NAN; *v = finite ? fma(fy, yd, v0) : NAN;
}
static void undistort_tail(const double* k, double fx, double fy, double u0, double v0, double X, double Y, double Wh, double* u, double* v) {
    const double w = 1. / Wh, x = X * w, y = Y * w;
    const double x2 = x * x, y2 = y * y, r2 = x2 + y2, _2xy = 2 * x * y, kr = cv_kr(k, r2);
    const double xd = fma(k[3], r2 + 2 * x2, fma(x, kr, k[2] * _2xy));
    const double yd = fma(k[3], _2xy, fma(y, kr, k[2] * (r2 + 2 * y2)));
    const int finite = isfinite(r2) && isfinite(xd) && isfinite(yd);
    *u = finite ? fma(fx, xd, u0) : NAN; *v = finite ? fma(fy, yd, v0) : NAN;
}

/* the int16 map of cv::undistort: per pixel sx, sy and the fraction index (iv & 31) * 32 + (iu & 31), as CV_16SC2 + CV_16UC1 */
VO_API int vo_undistort_map(int W, int H, const double* K, const double* dist, int n_dist, int16_t* sxy, uint16_t* frac) {
    if (n_dist != 4 && n_dist != 5 && n_dist != 8) return -1;
    if (W < 1 || H < 1 || W >= 32767 || H >= 32767) return -1;
    double k[8] = {0, 0, 0, 0, 0, 0, 0, 0};  /* k1 k2 p1 p2 k3 k4 k5 k6 */
    for (int i = 0; i < n_dist; i++) k[i] = dist[i];
    const double fx = K[0], fy = K[4], u0 = K[2], v0 = K[5];
    const int W8 = W - W % 8;
    int stripe0 = (1 << 12) / W;
    if (stripe0 < 1) stripe0 = 1;
    if (stripe0 > H) stripe0 = H;
    for (int y0 = 0; y0 < H; y0 += stripe0) {
        int n = stripe0 < H - y0 ? stripe0 : H - y0;
        double Ar[9], ir[9];
        memcpy(Ar, K, sizeof Ar);
        Ar[5] = v0 - y0;
        inv3x3_cv(Ar, ir);
        for (int i = 0; i < n; i++) {
            double X = fma(i, ir[1], ir[2]), Y = fma(i, ir[4], ir[5]), Wh = fma(i, ir[7], ir[8]);
            for (int j = 0; j < W; j++) {
                double u, v;
                const int body = j < W8;
                if (body) {
                    const int l = j % 8;
                    undistort_body(k, fx, fy, u0, v0, X + ir[0] * l, Y + ir[3] * l, Wh + ir[6] * l, &u, &v);
                    if (l == 7) { X += 8 * ir[0]; Y += 8 * ir[3]; Wh += 8 * ir[6]; }
                } else {
                    undistort_tail(k, fx, fy, u0, v0, X, Y, Wh, &u, &v);
                    X += ir[0]; Y += ir[3]; Wh += ir[6];
                }
                const int iu = cv_round(u * 32), iv = cv_round(v * 32);
                int sx = iu >> 5, sy = iv >> 5;
                if (body) { sx = sx < -32768 ? -32768 : (sx > 32767 ? 32767 : sx); sy = sy < -32768 ? -32768 : (sy > 32767 ? 32767 : sy); }
                const size_t o = (size_t)(y0 + i) * W + j;
                sxy[o * 2] = (int16_t)sx; sxy[o * 2 + 1] = (int16_t)sy;  /* the tail's (short) cast wraps */
                frac[o] = (uint16_t)((iv & 31) * 32 + (iu & 31));
            }
        }
    }
    return 0;
}

VO_API int vo_undistort(int W, int H, const uint8_t* src, const double* K, const double* dist, int n_dist, uint8_t* dst) {
    int16_t* sxy = malloc((size_t)W * H * 2 * sizeof(int16_t));
    uint16_t* frac = malloc((size_t)W * H * sizeof(uint16_t));
    int rc = sxy && frac ? vo_undistort_map(W, H, K, dist, n_dist, sxy, frac) : -2;
    if (rc == 0)
        for (size_t o = 0; o < (size_t)W * H; o++) {  /* remap INTER_LINEAR, BORDER_CONSTANT(0) */
            const int sx = sxy[o * 2], sy = sxy[o * 2 + 1], ax = frac[o] & 31, ay = frac[o] >> 5;
            const int wt[4] = {(32 - ax) * (32 - ay) * 32, ax * (32 - ay) * 32, (32 - ax) * ay * 32, ax * ay * 32};
            for (int c = 0; c < 3; c++) {
                int acc = 0;
                for (int t = 0; t < 4; t++) {
                    const int xx = sx + (t & 1), yy = sy + (t >> 1);
                    acc += ((xx >= 0 && xx < W && yy >= 0 && yy < H) ? src[((size_t)yy * W + xx) * 3 + c] : 0) * wt[t];
                }
                acc = (acc + (1 << 14)) >> 15;
                dst[o * 3 + c] = (uint8_t)(acc < 0 ? 0 : (acc > 255 ? 255 : acc));
            }
        }
    free(sxy); free(frac);
    return rc;
}
