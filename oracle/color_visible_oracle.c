/*
 * color_visible_oracle.c — CPU restatement of occlusion-aware colouring (vc_color_visible, include/voxcarve.h).
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT, like voxcarve_oracle.c (whose pinned reference arithmetic this file leaves untouched; the
 * projection and the colour bodies below are restated the same way).  The definition, step by step, for every surface voxel
 * (x, y, z) (occupied && !isInner, ascending flatten index) and every view v:
 *   1. sample points: the voxel and its 8 corners (x +- 1/2, y +- 1/2, z +- 1/2); w = (fl(y' s), fl(x' s), fl(-z' s), 1);
 *      projection: f64 sequential accumulation rounded once to f32 p0, p1, p2; u = p0 / p2, v = p1 / p2 in IEEE f32;
 *   2. eligible iff all 9 points have p2 > 0 and finite u, v;
 *   3. key = min p2; rectangle [round(min u), round(max u)] x [round(min v), round(max v)], half away from zero, clipped to
 *      the image (clamped in float before the conversion);
 *   4. zbuf[v] = min over the eligible pairs and the pixels of their rectangles, from +inf;
 *   5. observation iff eligible, the centre's pixel (the reference's) inside the image, and key <= fl(zbuf + fl(tolerance s));
 *   6. reconstructClosestColor (mode 1) / reconstructAvgColor (mode 2) over the observations only, in view order.
 * Build: gcc -O2 -ffp-contract=off (oracle/color_visible.py).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define VO_API __attribute__((visibility("default")))

/* VoxelCarving.cpp:19 second product, as vo_project in voxcarve_oracle.c */
static void project(const float* P, const float* w, float* proj) {
    for (int i = 0; i < 3; i++) {
        double s = (double)P[i * 4 + 0] * (double)w[0];
        s = s + (double)P[i * 4 + 1] * (double)w[1];
        s = s + (double)P[i * 4 + 2] * (double)w[2];
        s = s + (double)P[i * 4 + 3] * (double)w[3];
        proj[i] = (float)s;
    }
}

static int32_t round_to_int(float v) { /* (int)std::round(float), INT_MIN outside int range (vo_round_to_int) */
    float r = roundf(v);
    if (!(r >= -2147483648.0f && r < 2147483648.0f)) return INT32_MIN;
    return (int32_t)r;
}

static int round_clamped(float c, int n) { /* round half away from zero of c clamped to [-1, n] in float */
    const float t = c < -1.0f ? -1.0f : (c > (float)n ? (float)n : c);
    return (int)roundf(t);
}

static int getbit(const uint32_t* w, int X, int Y, int Z, int x, int y, int z) {
    if (x < 0 || x >= X || y < 0 || y >= Y || z < 0 || z >= Z) return 0;
    int Wx = (X + 31) / 32;
    return (w[((size_t)z * Y + y) * Wx + (x >> 5)] >> (x & 31)) & 1u;
}

typedef struct {
    int eligible, centre_in, px, py, x0, x1, y0, y1;
    float key;
} pair_t;

static pair_t vis_pair(const float* P, int x, int y, int z, float s, int W, int H) {
    pair_t q;
    memset(&q, 0, sizeof q);
    q.eligible = 1;
    float umin = 0, umax = 0, vmin = 0, vmax = 0;
    for (int c = 0; c < 9; c++) {
        float xp = (float)x, yp = (float)y, zp = (float)z;
        if (c > 0) {
            xp = xp + (((c - 1) & 1) ? 0.5f : -0.5f);
            yp = yp + (((c - 1) & 2) ? 0.5f : -0.5f);
            zp = zp + (((c - 1) & 4) ? 0.5f : -0.5f);
        }
        const float w[4] = {yp * s, xp * s, -zp * s, 1.0f}; /* Model.h:134-136 with the index as an f32 */
        float p[3];
        project(P, w, p);
        const float u = p[0] / p[2], v = p[1] / p[2];
        if (!(p[2] > 0.0f && isfinite(u) && isfinite(v))) q.eligible = 0;
        if (c == 0) {
            q.px = round_to_int(u);
            q.py = round_to_int(v);
            q.centre_in = q.px >= 0 && q.px < W && q.py >= 0 && q.py < H; /* VoxelCarving.cpp:44-45 */
            q.key = p[2];
            umin = umax = u;
            vmin = vmax = v;
        } else {
            if (p[2] < q.key) q.key = p[2];
            if (u < umin) umin = u;
            if (u > umax) umax = u;
            if (v < vmin) vmin = v;
            if (v > vmax) vmax = v;
        }
    }
    if (!q.eligible) return q; /* u, v may be NaN: no rectangle */
    q.x0 = round_clamped(umin, W); if (q.x0 < 0) q.x0 = 0;
    q.x1 = round_clamped(umax, W); if (q.x1 > W - 1) q.x1 = W - 1;
    q.y0 = round_clamped(vmin, H); if (q.y0 < 0) q.y0 = 0;
    q.y1 = round_clamped(vmax, H); if (q.y1 > H - 1) q.y1 = H - 1;
    return q;
}

/* Records as vo_color writes them (idx, rgbn = r, g, b, min(n_obs, 255); MODEL_COLOR with n = 0); obs_out (optional,
 * n_records * V bytes, [record][view]) receives the observation flags.  Returns the record count (records beyond cap are
 * counted, not written); UINT64_MAX if memory runs out. */
VO_API uint64_t vo_color_visible(int X, int Y, int Z, float s, int V, int W, int H, const float* P, const float* M,
                                 const uint8_t* images_bgr, const uint32_t* occ, int mode, float tolerance, uint64_t* idx_out,
                                 uint8_t* rgbn_out, uint8_t* obs_out, uint64_t cap) {
    uint64_t n = 0, n_alloc = 1024;
    int32_t* xyz = malloc(n_alloc * 3 * sizeof(int32_t));
    if (!xyz) return UINT64_MAX;
    for (int z = 0; z < Z; z++)
        for (int y = 0; y < Y; y++)
            for (int x = 0; x < X; x++) {
                if (!getbit(occ, X, Y, Z, x, y, z)) continue;
                int inner = getbit(occ, X, Y, Z, x - 1, y, z) && getbit(occ, X, Y, Z, x + 1, y, z) &&
                            getbit(occ, X, Y, Z, x, y - 1, z) && getbit(occ, X, Y, Z, x, y + 1, z) &&
                            getbit(occ, X, Y, Z, x, y, z - 1) && getbit(occ, X, Y, Z, x, y, z + 1); /* Model.h:126-132 */
                if (inner) continue;
                if (n == n_alloc) {
                    n_alloc *= 2;
                    int32_t* t = realloc(xyz, n_alloc * 3 * sizeof(int32_t));
                    if (!t) { free(xyz); return UINT64_MAX; }
                    xyz = t;
                }
                xyz[n * 3] = x; xyz[n * 3 + 1] = y; xyz[n * 3 + 2] = z;
                n++;
            }
    const float tau = tolerance * s;
    uint8_t* obs = calloc(n * (size_t)V + 1, 1);
    float* zbuf = malloc((size_t)W * H * sizeof(float));
    pair_t* pairs = malloc((n + 1) * sizeof(pair_t));
    if (!obs || !zbuf || !pairs) { free(xyz); free(obs); free(zbuf); free(pairs); return UINT64_MAX; }
    for (int v = 0; v < V; v++) {
        const float* Pv = P + (size_t)v * 12;
        for (size_t k = 0; k < (size_t)W * H; k++) zbuf[k] = INFINITY;
        for (uint64_t i = 0; i < n; i++) {
            pair_t q = vis_pair(Pv, xyz[i * 3], xyz[i * 3 + 1], xyz[i * 3 + 2], s, W, H);
            pairs[i] = q;
            if (!q.eligible) continue;
            for (int py = q.y0; py <= q.y1; py++)
                for (int px = q.x0; px <= q.x1; px++) {
                    float* d = zbuf + (size_t)py * W + px;
                    if (q.key < *d) *d = q.key;
                }
        }
        for (uint64_t i = 0; i < n; i++) {
            const pair_t* q = &pairs[i];
            if (q->eligible && q->centre_in && q->key <= zbuf[(size_t)q->py * W + q->px] + tau) obs[i * V + v] = 1;
        }
    }
    for (uint64_t i = 0; i < n; i++) {
        const int x = xyz[i * 3], y = xyz[i * 3 + 1], z = xyz[i * 3 + 2];
        const float w[4] = {(float)y * s, (float)x * s, (float)(-1 * z) * s, 1.0f}; /* vo_world */
        int nobs = 0;
        float sum[3] = {0, 0, 0}, best[3] = {50, 168, 141}, bestd = 0;
        for (int v = 0; v < V; v++) {
            if (!obs[i * V + v]) continue;
            const pair_t q = vis_pair(P + (size_t)v * 12, x, y, z, s, W, H); /* the centre pixel, inside the image */
            const uint8_t* pix = images_bgr + (((size_t)v * H + q.py) * W + q.px) * 3;
            float rgb[3] = {(float)pix[2], (float)pix[1], (float)pix[0]}; /* ColorReconstruction.h:59 BGR->RGB */
            const float cam[4] = {M[v * 12 + 3], M[v * 12 + 7], M[v * 12 + 11], 1.0f};
            double acc = 0; /* vo_depth: cv::norm(cam - w) */
            for (int k = 0; k < 4; k++) {
                float d = cam[k] - w[k];
                acc += (double)d * (double)d;
            }
            const float d = (float)sqrt(acc);
            if (nobs == 0 || d < bestd) { bestd = d; memcpy(best, rgb, sizeof best); } /* .cpp:34-40 */
            for (int c = 0; c < 3; c++) sum[c] = sum[c] + rgb[c];                     /* .cpp:60-64 */
            nobs++;
        }
        uint8_t out[4] = {50, 168, 141, (uint8_t)(nobs > 255 ? 255 : nobs)};
        if (nobs > 0)
            for (int c = 0; c < 3; c++) out[c] = (uint8_t)(mode == 2 ? roundf(sum[c] / (float)nobs) : best[c]);
        if (i < cap) {
            idx_out[i] = (uint64_t)x + (uint64_t)X * ((uint64_t)y + (uint64_t)Y * (uint64_t)z);
            memcpy(rgbn_out + i * 4, out, 4);
            if (obs_out) memcpy(obs_out + i * V, obs + i * V, V);
        }
    }
    free(xyz); free(obs); free(zbuf); free(pairs);
    return n;
}
