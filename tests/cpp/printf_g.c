/* printf("%g\n") of floats with the C library: the reference text for vc_format_g (tests/test_mesh_off.py,
 * tools/format_g_exhaustive.py).  Every thread formats a contiguous range into its own stretch of `out` (13 bytes per value:
 * at most 12 characters and the newline), then the stretches are moved together. */
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

typedef struct {
    const float* v;
    uint64_t n;
    char* out;
    uint64_t len;
} Part;

static void* run(void* arg) {
    Part* p = (Part*)arg;
    char line[32];
    uint64_t len = 0;
    for (uint64_t i = 0; i < p->n; i++) {
        const int k = snprintf(line, sizeof line, "%g\n", (double)p->v[i]);
        memcpy(p->out + len, line, (size_t)k);
        len += (uint64_t)k;
    }
    p->len = len;
    return NULL;
}

/* out must hold 13 n bytes; returns the length of the text */
uint64_t ref_format_g(const float* v, uint64_t n, char* out, int threads) {
    enum { MAXT = 256 };
    Part parts[MAXT];
    pthread_t th[MAXT];
    if (threads < 1) threads = 1;
    if (threads > MAXT) threads = MAXT;
    const uint64_t per = (n + (uint64_t)threads - 1) / (uint64_t)threads;
    for (int t = 0; t < threads; t++) {
        const uint64_t b = per * (uint64_t)t < n ? per * (uint64_t)t : n, e = b + per < n ? b + per : n;
        parts[t].v = v + b;
        parts[t].n = e - b;
        parts[t].out = out + 13 * b;
        parts[t].len = 0;
        pthread_create(&th[t], NULL, run, &parts[t]);
    }
    uint64_t pos = 0;
    for (int t = 0; t < threads; t++) {
        pthread_join(th[t], NULL);
        memmove(out + pos, parts[t].out, parts[t].len);
        pos += parts[t].len;
    }
    return pos;
}
