/* TEST INFRASTRUCTURE ONLY (oracle/): CPU restatement of the reference's per-pixel hot path.
 * See port.h.  Build: gcc -O2 -std=c11 -ffp-contract=off (oracle/Makefile) — the reference's
 * canonical semantics are "no FMA contraction" (SURVEY.md §0.7).
 *
 * Pinning status: every function below is checked against the reference's own compiled sources
 * (oracle/_ref/libvrt_ref*.so) in tests/test_oracle_pinned.py, except
 *   - gi_bounces == 2, vo_grid_render (mirror reflections) and the Philox lattice RNG: extensions with no
 *     reference behaviour ("parity unpinned" for those, specified in DESIGN.md §2).  gi_bounces == 1 follows the
 *     reference expression; feeding both sides the same random numbers is impossible with the reference's racy
 *     global RNG, so that pin is statistical (PSNR of images, tests/test_oracle_pinned.py);
 *   - vo_present (main.cpp:159-177): the reference blends through SFML/OpenGL, absent here — "parity unpinned", the
 *     arithmetic is round-to-nearest 8-bit unorm blending; the checkerboard / temporal blend that feeds it IS pinned
 *     (the reference's RayCaster driven by the main.cpp loop, tests/test_oracle_pinned.py, tests/golden/frame_checker_small.npz);
 *   - rays with a non-finite origin or direction: the reference never returns for them; defined here as a miss of
 *     complexity 0 (lsvo_cast_one);
 *   - glm itself is un-vendored and unpinned in the reference; the shim restates its public
 *     definitions (oracle/shim/glm/glm.hpp).
 */
#define _GNU_SOURCE
#include "port.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------------------------ */
/* helpers: src/utils.cpp                                                                      */
/* ------------------------------------------------------------------------------------------ */
static inline uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }   /* utils.cpp:109-112 */
static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }      /* utils.cpp:115-118 */
static inline float fracf_(float f) { float w; return modff(f, &w); }               /* utils.cpp:60-64  */
/* std::max / std::min as the reference uses them: max(a,b) = a<b ? b : a, min(a,b) = b<a ? b : a */
static inline float maxf_(float a, float b) { return a < b ? b : a; }
static inline float minf_(float a, float b) { return b < a ? b : a; }

typedef struct { float x, y, z; } v3;
static inline v3 v3_(float x, float y, float z) { v3 r = {x, y, z}; return r; }
static inline float dot3(v3 a, v3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }   /* glm::dot */
static inline v3 norm3(v3 v) {                                                      /* glm::normalize */
    const float inv = 1.0f / sqrtf(dot3(v, v));
    return v3_(v.x * inv, v.y * inv, v.z * inv);
}

/* ------------------------------------------------------------------------------------------ */
/* threading: contiguous blocks of work handed out round-robin                                  */
/* ------------------------------------------------------------------------------------------ */
typedef void (*range_fn)(void* ctx, uint64_t begin, uint64_t end);
typedef struct { range_fn fn; void* ctx; uint64_t n, block; int id, total; } par_arg;
static void* par_thread(void* a_) {
    par_arg* a = (par_arg*)a_;
    for (uint64_t b = (uint64_t)a->id * a->block; b < a->n; b += (uint64_t)a->total * a->block) {
        uint64_t e = b + a->block < a->n ? b + a->block : a->n;
        a->fn(a->ctx, b, e);
    }
    return NULL;
}
static void par_for(range_fn fn, void* ctx, uint64_t n, uint64_t block, int threads) {
    if (threads <= 1) { fn(ctx, 0, n); return; }
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)threads);
    par_arg* args = (par_arg*)malloc(sizeof(par_arg) * (size_t)threads);
    for (int i = 0; i < threads; ++i) {
        par_arg a = {fn, ctx, n, block, i, threads};
        args[i] = a;
        pthread_create(&th[i], NULL, par_thread, &args[i]);
    }
    for (int i = 0; i < threads; ++i) pthread_join(th[i], NULL);
    free(th); free(args);
}

/* ------------------------------------------------------------------------------------------ */
/* FastNoise 0.4.1, 2-D SimplexFractal FBM: lib/fastnoise/FastNoise.cpp:197-215 (SetSeed),     */
/* :217-227 (fractal bounding), :410-447 (GetNoise), :1191-1207 (FBM), :1275-1333 (simplex).   */
/* std::mt19937_64 is restated from its ISO C++ definition (MT19937-64, Matsumoto/Nishimura).   */
/* ------------------------------------------------------------------------------------------ */
static uint8_t g_perm[512], g_perm12[512];
static int g_perm_ready = 0;
static pthread_mutex_t g_perm_lock = PTHREAD_MUTEX_INITIALIZER;

static void noise_seed(uint64_t seed) {
    enum { NN = 312, MM = 156 };
    static uint64_t mt[NN];
    mt[0] = seed;
    for (int i = 1; i < NN; ++i) mt[i] = 6364136223846793005ULL * (mt[i - 1] ^ (mt[i - 1] >> 62)) + (uint64_t)i;
    int idx = NN;
    for (int i = 0; i < 256; ++i) g_perm[i] = (uint8_t)i;
    for (int j = 0; j < 256; ++j) {
        if (idx >= NN) {
            for (int i = 0; i < NN; ++i) {
                const uint64_t x = (mt[i] & 0xFFFFFFFF80000000ULL) | (mt[(i + 1) % NN] & 0x7FFFFFFFULL);
                mt[i] = mt[(i + MM) % NN] ^ (x >> 1) ^ ((x & 1ULL) ? 0xB5026F5AA96619E9ULL : 0ULL);
            }
            idx = 0;
        }
        uint64_t y = mt[idx++];
        y ^= (y >> 29) & 0x5555555555555555ULL;
        y ^= (y << 17) & 0x71D67FFFEDA60000ULL;
        y ^= (y << 37) & 0xFFF7EEE000000000ULL;
        y ^= (y >> 43);
        const int k = (int)(y % (uint64_t)(256 - j)) + j;
        const uint8_t l = g_perm[j];
        g_perm[j] = g_perm[j + 256] = g_perm[k];
        g_perm[k] = l;
        g_perm12[j] = g_perm12[j + 256] = (uint8_t)(g_perm[j] % 12);
    }
}
static void noise_init(void) {
    pthread_mutex_lock(&g_perm_lock);
    if (!g_perm_ready) { noise_seed(1337); g_perm_ready = 1; }
    pthread_mutex_unlock(&g_perm_lock);
}

static const float GX[12] = {1, -1, 1, -1, 1, -1, 1, -1, 0, 0, 0, 0};
static const float GY[12] = {1, 1, -1, -1, 0, 0, 0, 0, 1, -1, 1, -1};

static inline int ffloor_(float f) { return f >= 0 ? (int)f : (int)f - 1; }
static inline float grad2(uint8_t off, int x, int y, float xd, float yd) {
    const uint8_t l = g_perm12[(x & 0xff) + g_perm[(y & 0xff) + off]];
    return xd * GX[l] + yd * GY[l];
}
static float simplex2(uint8_t off, float x, float y) {
    const float SQRT3 = 1.7320508075688772935274463415059f;
    const float F2 = 0.5f * (SQRT3 - 1.0f);
    const float G2 = (3.0f - SQRT3) / 6.0f;
    float t = (x + y) * F2;
    const int i = ffloor_(x + t), j = ffloor_(y + t);
    t = (float)(i + j) * G2;
    const float X0 = (float)i - t, Y0 = (float)j - t;
    const float x0 = x - X0, y0 = y - Y0;
    const int i1 = x0 > y0 ? 1 : 0, j1 = 1 - i1;
    const float x1 = x0 - (float)i1 + G2, y1 = y0 - (float)j1 + G2;
    const float x2 = x0 - 1 + 2 * G2, y2 = y0 - 1 + 2 * G2;
    float n0 = 0, n1 = 0, n2 = 0;
    t = 0.5f - x0 * x0 - y0 * y0;
    if (!(t < 0)) { t *= t; n0 = t * t * grad2(off, i, j, x0, y0); }
    t = 0.5f - x1 * x1 - y1 * y1;
    if (!(t < 0)) { t *= t; n1 = t * t * grad2(off, i + i1, j + j1, x1, y1); }
    t = 0.5f - x2 * x2 - y2 * y2;
    if (!(t < 0)) { t *= t; n2 = t * t * grad2(off, i + 1, j + 1, x2, y2); }
    return 70 * (n0 + n1 + n2);
}
float vo_noise2d(float x, float y) {
    noise_init();
    const float frequency = 0.01f, lacunarity = 2.0f, gain = 0.5f;
    const int octaves = 3;
    float amp = gain, amp_fractal = 1.0f;
    for (int i = 1; i < octaves; ++i) { amp_fractal += amp; amp *= gain; }
    const float bounding = 1.0f / amp_fractal;
    x *= frequency; y *= frequency;
    float sum = simplex2(g_perm[0], x, y);
    amp = 1;
    for (int i = 1; i < octaves; ++i) {
        x *= lacunarity; y *= lacunarity;
        amp *= gain;
        sum += simplex2(g_perm[i], x, y) * amp;
    }
    return sum * bounding;
}
void vo_terrain_heights(int32_t size, int32_t* out) {           /* main.cpp:63-68 */
    for (uint32_t x = 0; x < (uint32_t)size; ++x)
        for (uint32_t z = 0; z < (uint32_t)size; ++z)
            out[(size_t)x * (size_t)size + z] = (int32_t)(64.0f * vo_noise2d(0.75f * (float)x, 0.75f * (float)z) + 32);
}

/* ------------------------------------------------------------------------------------------ */
/* compileSVO without the pointer tree: lsvo_utils.cpp:4-49                                    */
/* ------------------------------------------------------------------------------------------ */
typedef struct builder {
    vo_lnode* out; uint64_t cap, count;
    int S;
    /* terrain mode: top[l][(x>>l)*(S>>l)+(z>>l)] = highest solid y over the 2^l square, bottom is S/2+1 */
    int32_t** top; int bottom;
    /* dense mode: occ[l] occupancy pyramid, occ[l][((x>>l)*(S>>l)+(y>>l))*(S>>l)+(z>>l)] */
    uint8_t** occ;
} builder;

static int cube_nonempty(const builder* b, int l, int x0, int y0, int z0) {   /* cube of edge 2^l */
    const int n = b->S >> l;
    if (b->top) {
        const int32_t t = b->top[l][(size_t)(x0 >> l) * (size_t)n + (size_t)(z0 >> l)];
        return t >= y0 && y0 + (1 << l) - 1 >= b->bottom && t >= b->bottom;
    }
    return b->occ[l][((size_t)(x0 >> l) * (size_t)n + (size_t)(y0 >> l)) * (size_t)n + (size_t)(z0 >> l)] != 0;
}
static void slot_default(builder* b, uint64_t i) {      /* LNode(), lsvo_utils.hpp:7-12 */
    if (b->out && i < b->cap) { vo_lnode d = {1, 0, 0, 0, 0}; b->out[i] = d; }
}
/* node `idx` covers the cube of edge 2^l at (x0,y0,z0), l >= 1 */
static void build_rec(builder* b, uint64_t idx, int l, int x0, int y0, int z0) {
    const uint64_t child_pos = b->count;                              /* :7  */
    if (b->out && idx < b->cap) b->out[idx].child_offset = (uint32_t)(child_pos - idx);   /* :8-10 */
    const int h = 1 << (l - 1);
    int any = 0;
    for (int c = 0; c < 8 && !any; ++c)
        any = cube_nonempty(b, l - 1, x0 + (c & 1) * h, y0 + ((c >> 1) & 1) * h, z0 + ((c >> 2) & 1) * h);
    if (!any) return;                                                  /* :12-23 */
    for (int i = 0; i < 8; ++i) slot_default(b, b->count++);          /* :25-27 */
    for (int cx = 0; cx < 2; ++cx)                                     /* :29-31, x outer … z inner */
        for (int cy = 0; cy < 2; ++cy)
            for (int cz = 0; cz < 2; ++cz) {
                const int x1 = x0 + cx * h, y1 = y0 + cy * h, z1 = z0 + cz * h;
                if (!cube_nonempty(b, l - 1, x1, y1, z1)) continue;
                const int sub = cz * 4 + cy * 2 + cx;                  /* :34 */
                if (b->out && idx < b->cap) b->out[idx].child_mask |= (uint8_t)(1u << sub);
                if (l - 1 == 0) {                                      /* leaf: :40-42 */
                    if (b->out && idx < b->cap) b->out[idx].leaf_mask |= (uint8_t)(1u << sub);
                } else {
                    build_rec(b, child_pos + (uint64_t)sub, l - 1, x1, y1, z1);   /* :37-39 */
                }
            }
}
static uint64_t build_run(builder* b, int depth) {
    b->count = 0;
    slot_default(b, b->count++);                                       /* lsvo_utils.hpp:49 */
    build_rec(b, 0, depth, 0, 0, 0);
    return b->count;
}

uint64_t vo_build_terrain_lsvo(int depth, const int32_t* heights, vo_lnode* out, uint64_t cap) {
    const int S = 1 << depth;
    builder b; memset(&b, 0, sizeof(b));
    b.out = out; b.cap = cap; b.S = S; b.bottom = S / 2 + 1;
    b.top = (int32_t**)calloc((size_t)depth + 1, sizeof(int32_t*));
    b.top[0] = (int32_t*)malloc(sizeof(int32_t) * (size_t)S * (size_t)S);
    for (size_t i = 0; i < (size_t)S * (size_t)S; ++i) {
        int32_t hm = heights[i] < S ? heights[i] : S;                  /* main.cpp:72: max(16, min(S, h)) */
        if (hm < 16) hm = 16;
        b.top[0][i] = S / 2 + hm - 1;                                  /* y in [1,hm) → y + S/2 */
    }
    for (int l = 1; l <= depth; ++l) {
        const int n = S >> l, m = S >> (l - 1);
        b.top[l] = (int32_t*)malloc(sizeof(int32_t) * (size_t)n * (size_t)n);
        for (int x = 0; x < n; ++x)
            for (int z = 0; z < n; ++z) {
                int32_t t = b.top[l - 1][(size_t)(2 * x) * m + 2 * z];
                const int32_t t1 = b.top[l - 1][(size_t)(2 * x) * m + 2 * z + 1];
                const int32_t t2 = b.top[l - 1][(size_t)(2 * x + 1) * m + 2 * z];
                const int32_t t3 = b.top[l - 1][(size_t)(2 * x + 1) * m + 2 * z + 1];
                if (t1 > t) t = t1;
                if (t2 > t) t = t2;
                if (t3 > t) t = t3;
                b.top[l][(size_t)x * n + z] = t;
            }
    }
    const uint64_t cnt = build_run(&b, depth);
    for (int l = 0; l <= depth; ++l) free(b.top[l]);
    free(b.top);
    return cnt;
}

static uint8_t** occ_pyramid(int depth, const uint8_t* occ) {
    const int S = 1 << depth;
    uint8_t** p = (uint8_t**)calloc((size_t)depth + 1, sizeof(uint8_t*));
    p[0] = (uint8_t*)malloc((size_t)S * S * S);
    for (size_t i = 0; i < (size_t)S * S * S; ++i) p[0][i] = occ[i] != 0;
    for (int l = 1; l <= depth; ++l) {
        const size_t n = (size_t)(S >> l), m = (size_t)(S >> (l - 1));
        p[l] = (uint8_t*)calloc(n * n * n, 1);
        for (size_t x = 0; x < m; ++x)
            for (size_t y = 0; y < m; ++y)
                for (size_t z = 0; z < m; ++z)
                    if (p[l - 1][(x * m + y) * m + z]) p[l][((x >> 1) * n + (y >> 1)) * n + (z >> 1)] = 1;
    }
    return p;
}
static void occ_pyramid_free(uint8_t** p, int depth) {
    for (int l = 0; l <= depth; ++l) free(p[l]);
    free(p);
}

uint64_t vo_build_dense_lsvo(int depth, const uint8_t* occ, vo_lnode* out, uint64_t cap) {
    builder b; memset(&b, 0, sizeof(b));
    b.out = out; b.cap = cap; b.S = 1 << depth;
    b.occ = occ_pyramid(depth, occ);
    const uint64_t cnt = build_run(&b, depth);
    occ_pyramid_free(b.occ, depth);
    return cnt;
}

/* ------------------------------------------------------------------------------------------ */
/* LSVO<D>::castRay, include/lsvo.hpp:33-172                                                   */
/* ------------------------------------------------------------------------------------------ */
static void lsvo_cast_one(const vo_lnode* nodes, int depth, int guard, const float o[3], const float din[3],
                          float coef, float bias, vo_hit* res) {
    const float EPS = 1.0f / (float)(1 << 23);                        /* :40 */
    const int depth_offset = 23 - depth;                              /* :38 */
    uint32_t stack_parent[24]; float stack_tmax[24];                  /* :42 (MAX_DEPTH+1 entries) */
    float d[3], tc[3], to[3], p[3];
    uint32_t mirror = 7u;
    memset(res, 0, sizeof(*res));
    /* A ray with a non-finite origin or direction never leaves the reference's loop (comparisons with NaN all fail:
     * no descent, no step, no pop).  The engine and this restatement define it as a miss of complexity 0. */
    /* x * 0 is NaN exactly for infinite / NaN x: tested per component, so that finite rays whose components would overflow a sum stay finite */
    if ((((o[0] * 0.0f + o[1] * 0.0f) + o[2] * 0.0f) + ((din[0] * 0.0f + din[1] * 0.0f) + din[2] * 0.0f)) != 0.0f) return;
    for (int a = 0; a < 3; ++a) {
        d[a] = din[a];
        if (fabsf(d[a]) < EPS) d[a] = copysignf(EPS, d[a]);           /* :44-46 */
        tc[a] = -1.0f / fabsf(d[a]);                                  /* :47 */
        to[a] = o[a] * tc[a];                                         /* :48 */
        if (d[a] > 0.0f) { mirror ^= 1u << a; to[a] = 3.0f * tc[a] - to[a]; }   /* :50-52 */
    }
    float t_min = maxf_(2.0f * tc[0] - to[0], maxf_(2.0f * tc[1] - to[1], 2.0f * tc[2] - to[2]));   /* :54 */
    float t_max = minf_(tc[0] - to[0], minf_(tc[1] - to[1], tc[2] - to[2]));                       /* :55 */
    float h = t_max;
    t_min = maxf_(0.0f, t_min);                                       /* :57 */
    t_max = minf_(1.0f, t_max);                                       /* :58 */
    uint32_t parent = 0u, child = 0u, face = 0u;
    int scale = 22;                                                   /* int8_t in the reference (:62) */
    float scale_f = 0.5f;
    for (int a = 0; a < 3; ++a) {
        p[a] = 1.0f;
        if (1.5f * tc[a] - to[a] > t_min) { child ^= 1u << a; p[a] = 1.5f; }   /* :66-68 */
    }
    int hit = 0;
    uint32_t iters = 0;
    while (scale < 23 && scale > guard) {                             /* :72 */
        ++iters;
        const vo_lnode nd = nodes[parent];                            /* :74 */
        float corner[3];
        for (int a = 0; a < 3; ++a) corner[a] = p[a] * tc[a] - to[a]; /* :76 */
        const float tc_max = minf_(corner[0], minf_(corner[1], corner[2]));
        const uint32_t shift = child ^ mirror;                        /* :79 */
        if (((nd.child_mask >> shift) & 1u) && t_min <= t_max) {      /* :80-81 */
            if (tc_max * coef + bias >= scale_f) { hit = 1; break; }  /* :82-85 */
            const float tv_max = minf_(t_max, tc_max);
            const float half = scale_f * 0.5f;
            if (t_min <= tv_max) {                                    /* :89 */
                if ((nd.leaf_mask >> shift) & 1u) { hit = 1; break; } /* :90-95 */
                if (tc_max < h) {                                     /* :97-100 */
                    stack_parent[scale - depth_offset] = parent;
                    stack_tmax[scale - depth_offset] = t_max;
                }
                h = tc_max;
                parent += nd.child_offset + shift;                    /* :103 */
                child = 0u;
                --scale;
                scale_f = half;
                for (int a = 0; a < 3; ++a) {
                    const float t_half = half * tc[a] + corner[a];    /* :88 */
                    if (t_half > t_min) { child ^= 1u << a; p[a] += scale_f; }   /* :107-109 */
                }
                t_max = tv_max;
                continue;
            }
        }
        uint32_t step = 0u;                                           /* :115-118 */
        for (int a = 0; a < 3; ++a)
            if (corner[a] <= tc_max) { step ^= 1u << a; p[a] -= scale_f; }
        t_min = tc_max;
        child ^= step;
        face = step;
        if (child & step) {                                           /* :124-145 */
            uint32_t diff = 0u;
            uint32_t ip[3];
            for (int a = 0; a < 3; ++a) {
                ip[a] = f2u(p[a]);
                if (step & (1u << a)) diff |= ip[a] ^ f2u(p[a] + scale_f);
            }
            scale = (int)(int8_t)((f2u((float)diff) >> 23) - 127u);   /* :132 */
            scale_f = u2f((uint32_t)(scale - 23 + 127) << 23);        /* :133 */
            if (scale >= 23) break;       /* the reference reads the stack first; the value is unused */
            parent = stack_parent[scale - depth_offset];
            t_max = stack_tmax[scale - depth_offset];
            child = 0u;
            for (int a = 0; a < 3; ++a) {
                const uint32_t sh = ip[a] >> scale;
                p[a] = u2f(sh << scale);
                child |= (sh & 1u) << a;
            }
            h = 0.0f;
        }
    }
    res->complexity = iters;
    if (!hit) return;
    res->hit = 1;
    res->scale = scale;
    res->face = face;
    for (int a = 0; a < 3; ++a) {
        const float sg = (float)(0.0f < d[a]) - (float)(d[a] < 0.0f);            /* glm::sign */
        res->normal[a] = (-sg) * (float)(face & (1u << a));                       /* :149 */
        if ((mirror & (1u << a)) == 0) p[a] = 3.0f - scale_f - p[a];              /* :151-153 */
        res->position[a] = minf_(maxf_(o[a] + t_min * d[a], p[a] + EPS), p[a] + scale_f - EPS);   /* :156-158 */
        res->voxel[a] = (int32_t)((p[a] - 1.0f) * (float)(1 << depth));
    }
    res->distance = t_min;                                            /* :155 */
    const float S = (float)(1 << depth);                              /* :39 */
    if (res->normal[0] != 0.0f) {                                     /* :160-168 */
        res->voxel_coord[0] = fracf_(res->position[2] * S); res->voxel_coord[1] = fracf_(res->position[1] * S);
    } else if (res->normal[1] != 0.0f) {
        res->voxel_coord[0] = fracf_(res->position[0] * S); res->voxel_coord[1] = fracf_(res->position[2] * S);
    } else if (res->normal[2] != 0.0f) {
        res->voxel_coord[0] = fracf_(res->position[0] * S); res->voxel_coord[1] = fracf_(res->position[1] * S);
    }   /* else: uninitialised in the reference (ray started inside a solid cell); zero here */
}

typedef struct { const vo_lnode* nodes; int depth, guard; const float *o, *d; float coef, bias; vo_hit* out; } lsvo_ctx;
static void lsvo_range(void* c_, uint64_t b, uint64_t e) {
    lsvo_ctx* c = (lsvo_ctx*)c_;
    for (uint64_t i = b; i < e; ++i) lsvo_cast_one(c->nodes, c->depth, c->guard, c->o + 3 * i, c->d + 3 * i, c->coef, c->bias, c->out + i);
}
void vo_lsvo_cast(const vo_lnode* nodes, int depth, int guard, const float* origin, const float* dir, float coef,
                  float bias, uint64_t n, vo_hit* out, int threads) {
    lsvo_ctx c = {nodes, depth, guard, origin, dir, coef, bias, out};
    par_for(lsvo_range, &c, n, 4096, threads);
}

/* ------------------------------------------------------------------------------------------ */
/* The same walk with the structural changes of the device loop (csrc/lsvo_step.cuh, Trav2) — a CPU cross-check of the
 * arguments in DESIGN.md §4, NOT a second specification: tests/test_oracle_golden.py asserts that it returns exactly what
 * lsvo_cast_one returns (records and trip counts) on terrain, random voxel sets and degenerate rays.
 *   - the stack write of lsvo.hpp:97-100 is unconditional (no `h`);
 *   - cone hit (:82-85) and leaf hit (:90-95) share one exit; there is no hit flag: how the walk ended is read off its
 *     final state (a coordinate below 1 / the guard / otherwise a hit);
 *   - the guard test is dropped where it cannot bind (guard < 23 - depth);
 *   - the child selection uses fmaf(half, tc, c) when `unit` is set (exact product: half is a power of two);
 *   - the node is fetched when `parent` changes only.                                                                    */
static void lsvo_cast_one_restructured(const vo_lnode* nodes, int depth, int guard, const float o[3], const float din[3],
                                       float coef, float bias, int unit, vo_hit* res) {
    const float EPS = 1.0f / (float)(1 << 23);
    const int depth_offset = 23 - depth;
    const int guarded = guard >= 23 - depth;
    const float guard_sf = u2f((uint32_t)(guard + 104) << 23);
    uint32_t stack_parent[24]; float stack_tmax[24];
    float d[3], tc[3], to[3], p[3];
    uint32_t mirror = 7u;
    memset(res, 0, sizeof(*res));
    if ((((o[0] * 0.0f + o[1] * 0.0f) + o[2] * 0.0f) + ((din[0] * 0.0f + din[1] * 0.0f) + din[2] * 0.0f)) != 0.0f) return;
    for (int a = 0; a < 3; ++a) {
        d[a] = din[a];
        if (fabsf(d[a]) < EPS) d[a] = copysignf(EPS, d[a]);
        tc[a] = -1.0f / fabsf(d[a]);
        to[a] = o[a] * tc[a];
        if (d[a] > 0.0f) { mirror ^= 1u << a; to[a] = 3.0f * tc[a] - to[a]; }
    }
    float t_min = maxf_(2.0f * tc[0] - to[0], maxf_(2.0f * tc[1] - to[1], 2.0f * tc[2] - to[2]));
    float t_max = minf_(tc[0] - to[0], minf_(tc[1] - to[1], tc[2] - to[2]));
    t_min = maxf_(0.0f, t_min);
    t_max = minf_(1.0f, t_max);
    uint32_t parent = 0u, child = 0u, face = 0u;
    float sf = 0.5f;
    for (int a = 0; a < 3; ++a) {
        p[a] = 1.0f;
        if (1.5f * tc[a] - to[a] > t_min) { child ^= 1u << a; p[a] = 1.5f; }
    }
    uint32_t iters = 0;
    vo_lnode nd = nodes[0];
    if (guarded && !(sf > guard_sf)) { res->complexity = 0; return; }   /* the loop condition before the first trip (:72) */
    for (;;) {
        ++iters;
        float corner[3];
        for (int a = 0; a < 3; ++a) corner[a] = p[a] * tc[a] - to[a];
        const float tc_max = minf_(corner[0], minf_(corner[1], corner[2]));
        const uint32_t shift = child ^ mirror;
        if (((nd.child_mask >> shift) & 1u) && t_min <= t_max) {
            const float tv_max = minf_(t_max, tc_max);
            const int inside = t_min <= tv_max;
            int ends = inside && ((nd.leaf_mask >> shift) & 1u);
            if (tc_max * coef + bias >= sf) ends = 1;
            if (ends) break;
            if (inside) {
                const float half = sf * 0.5f;
                int scale = (int)(f2u(sf) >> 23) - 104;
                stack_parent[scale - depth_offset] = parent;
                stack_tmax[scale - depth_offset] = t_max;
                parent += nd.child_offset + shift;
                nd = nodes[parent];
                child = 0u;
                sf = half;
                for (int a = 0; a < 3; ++a) {
                    const float t_half = unit ? fmaf(half, tc[a], corner[a]) : half * tc[a] + corner[a];
                    if (t_half > t_min) { child ^= 1u << a; p[a] += half; }
                }
                t_max = tv_max;
                if (guarded && !(sf > guard_sf)) break;
                continue;
            }
        }
        uint32_t step = 0u;
        for (int a = 0; a < 3; ++a)
            if (corner[a] <= tc_max) { step ^= 1u << a; p[a] -= sf; }
        t_min = tc_max;
        child ^= step;
        face = step;
        if (child & step) {
            uint32_t diff = 0u, ip[3];
            for (int a = 0; a < 3; ++a) {
                ip[a] = f2u(p[a]);
                if (step & (1u << a)) diff |= ip[a] ^ f2u(p[a] + sf);
            }
            int scale = 31 - __builtin_clz(diff);
            if (scale >= 23) break;
            parent = stack_parent[scale - depth_offset];
            t_max = stack_tmax[scale - depth_offset];
            nd = nodes[parent];
            sf = u2f((uint32_t)(scale + 104) << 23);
            const uint32_t bit = 1u << scale, keep = 0u - bit;
            child = ((ip[0] & bit) + 2u * (ip[1] & bit) + 4u * (ip[2] & bit)) >> scale;
            for (int a = 0; a < 3; ++a) p[a] = u2f(ip[a] & keep);
            if (guarded && !(scale > guard)) break;
        }
    }
    res->complexity = iters;
    int miss = minf_(p[0], minf_(p[1], p[2])) < 1.0f;
    if (guarded && !(sf > guard_sf)) miss = 1;
    if (miss) return;
    const int scale = (int)(f2u(sf) >> 23) - 104;
    res->hit = 1;
    res->scale = scale;
    res->face = face;
    for (int a = 0; a < 3; ++a) {
        const float sg = (float)(0.0f < d[a]) - (float)(d[a] < 0.0f);
        res->normal[a] = (-sg) * (float)(face & (1u << a));
        if ((mirror & (1u << a)) == 0) p[a] = 3.0f - sf - p[a];
        res->position[a] = minf_(maxf_(o[a] + t_min * d[a], p[a] + EPS), p[a] + sf - EPS);
        res->voxel[a] = (int32_t)((p[a] - 1.0f) * (float)(1 << depth));
    }
    res->distance = t_min;
    const float S = (float)(1 << depth);
    if (res->normal[0] != 0.0f) {
        res->voxel_coord[0] = fracf_(res->position[2] * S); res->voxel_coord[1] = fracf_(res->position[1] * S);
    } else if (res->normal[1] != 0.0f) {
        res->voxel_coord[0] = fracf_(res->position[0] * S); res->voxel_coord[1] = fracf_(res->position[2] * S);
    } else if (res->normal[2] != 0.0f) {
        res->voxel_coord[0] = fracf_(res->position[0] * S); res->voxel_coord[1] = fracf_(res->position[1] * S);
    }
}
typedef struct { const vo_lnode* nodes; int depth, guard; const float *o, *d; float coef, bias; int unit; vo_hit* out; } lsvo2_ctx;
static void lsvo2_range(void* c_, uint64_t b, uint64_t e) {
    lsvo2_ctx* c = (lsvo2_ctx*)c_;
    for (uint64_t i = b; i < e; ++i)
        lsvo_cast_one_restructured(c->nodes, c->depth, c->guard, c->o + 3 * i, c->d + 3 * i, c->coef, c->bias, c->unit, c->out + i);
}
void vo_lsvo_cast_restructured(const vo_lnode* nodes, int depth, int guard, const float* origin, const float* dir, float coef,
                               float bias, int unit, uint64_t n, vo_hit* out, int threads) {
    lsvo2_ctx c = {nodes, depth, guard, origin, dir, coef, bias, unit, out};
    par_for(lsvo2_range, &c, n, 4096, threads);
}

/* ------------------------------------------------------------------------------------------ */
/* Grid3D<X,Y,Z>::castRay, include/grid_3d.hpp:35-132                                          */
/* ------------------------------------------------------------------------------------------ */
static void grid_cast_one(const uint8_t* cells, int X, int Y, int Z, const float o[3], const float d[3], vo_hit* res,
                          uint32_t* steps) {
    memset(res, 0, sizeof(*res));
    float td[3], tm[3];
    int st[3], c[3];
    const int dim[3] = {X, Y, Z};
    for (int a = 0; a < 3; ++a) {
        td[a] = fabsf(1.0f / d[a]);                                   /* :42-44 */
        st[a] = d[a] < 0 ? -1 : 1;                                    /* :48-50 */
        c[a] = (int)o[a];                                             /* :58-60 */
        tm[a] = ((float)(c[a] + (st[a] > 0 ? 1 : 0)) - o[a]) / d[a];  /* :62-64 */
    }
    int side = 0;
    uint32_t iter = 0;
    while (c[0] >= 0 && c[1] >= 0 && c[2] >= 0 && c[0] < X && c[1] < Y && c[2] < Z && iter < 2048u) {   /* :70 */
        float t;
        ++iter;
        if (tm[0] < tm[1]) side = tm[0] < tm[2] ? 0 : 2;              /* :73-99 */
        else side = tm[1] < tm[2] ? 1 : 2;
        t = tm[side];
        tm[side] += td[side];
        c[side] += st[side];
        if (c[0] >= 0 && c[1] >= 0 && c[2] >= 0 && c[0] < dim[0] && c[1] < dim[1] && c[2] < dim[2]) {   /* :101 */
            if (cells[((size_t)c[0] * (size_t)Y + (size_t)c[1]) * (size_t)Z + (size_t)c[2]] != 0) {      /* :103-104 */
                const float hx = o[0] + t * d[0], hy = o[1] + t * d[1], hz = o[2] + t * d[2];
                res->hit = 1;
                res->position[0] = hx; res->position[1] = hy; res->position[2] = hz;
                res->normal[side] = (float)(-st[side]);              /* :112-121 (others 0.0f) */
                if (side == 0) { res->voxel_coord[0] = 1.0f - fracf_(hz); res->voxel_coord[1] = fracf_(hy); }
                else if (side == 1) { res->voxel_coord[0] = fracf_(hx); res->voxel_coord[1] = fracf_(hz); }
                else { res->voxel_coord[0] = fracf_(hx); res->voxel_coord[1] = fracf_(hy); }
                res->distance = t;
                res->complexity = iter;                               /* :124 (only set on a hit) */
                res->face = 1u << side;
                res->voxel[0] = c[0]; res->voxel[1] = c[1]; res->voxel[2] = c[2];
                break;
            }
        }
    }
    if (steps) *steps = iter;
}
typedef struct { const uint8_t* cells; int X, Y, Z; const float *o, *d; vo_hit* out; uint32_t* steps; } grid_ctx;
static void grid_range(void* c_, uint64_t b, uint64_t e) {
    grid_ctx* c = (grid_ctx*)c_;
    for (uint64_t i = b; i < e; ++i)
        grid_cast_one(c->cells, c->X, c->Y, c->Z, c->o + 3 * i, c->d + 3 * i, c->out + i, c->steps ? c->steps + i : NULL);
}
void vo_grid_cast(const uint8_t* cells, int X, int Y, int Z, const float* origin, const float* dir, uint64_t n,
                  vo_hit* out, uint32_t* steps, int threads) {
    grid_ctx c = {cells, X, Y, Z, origin, dir, out, steps};
    par_for(grid_range, &c, n, 4096, threads);
}

/* ------------------------------------------------------------------------------------------ */
/* A conservative miss test for Grid3D::castRay on a coarse, dilated occupancy (DESIGN.md §7 (6): what a pyramid CAN do for
 * the dense grids without changing a record).  `coarse` holds one byte per cube of 2^shift cells: non-zero when the cube, or
 * any cube within two cubes of it on every axis, holds a solid cell.  The EXACT ray (double precision) is marched through the
 * coarse grid; if it meets no marked cube the reference's fp DDA — whose cells stay within one cell per axis of the exact ray's
 * cell, see the argument in DESIGN.md — cannot meet a solid cell either.  Returns 1 = certainly a miss, 0 = unknown (walk it).
 * Prototype and cross-check only (tests/test_oracle_golden.py); the product does not use it yet. */
static int grid_miss_one(const uint8_t* coarse, int CX, int CY, int CZ, int shift, int X, int Y, int Z, const float o[3],
                         const float d[3]) {
    const int dim[3] = {X, Y, Z}, cdim[3] = {CX, CY, CZ};
    double tm[3], td[3];
    int c[3], st[3];
    for (int a = 0; a < 3; ++a) {
        if (!(o[a] * 0.0f == 0.0f) || !(d[a] * 0.0f == 0.0f) || d[a] == 0.0f) return 0;   /* the fp walk of such a ray is not the ray */
        if (!(fabsf(o[a]) < 1.0e9f)) return 0;                                         /* (int)o would overflow */
        const int cell = (int)o[a];                                                    /* :58-60 */
        if (cell < 0 || cell >= dim[a] || o[a] < 0.0f) return (o[a] < 0.0f && cell == 0) ? 0 : 1;   /* starts outside: no trip, a miss */
        c[a] = cell >> shift;
        st[a] = d[a] < 0 ? -1 : 1;
        const double edge = (double)((c[a] + (st[a] > 0 ? 1 : 0)) << shift);
        td[a] = fabs((double)(1 << shift) / (double)d[a]);
        tm[a] = (edge - (double)o[a]) / (double)d[a];
    }
    for (;;) {
        if (coarse[((size_t)c[0] * (size_t)cdim[1] + (size_t)c[1]) * (size_t)cdim[2] + (size_t)c[2]]) return 0;
        const int side = tm[0] < tm[1] ? (tm[0] < tm[2] ? 0 : 2) : (tm[1] < tm[2] ? 1 : 2);
        tm[side] += td[side];
        c[side] += st[side];
        if (c[side] < 0 || c[side] >= cdim[side]) return 1;
    }
}
typedef struct { const uint8_t* coarse; int CX, CY, CZ, shift, X, Y, Z; const float *o, *d; uint8_t* out; } gmiss_ctx;
static void gmiss_range(void* c_, uint64_t b, uint64_t e) {
    gmiss_ctx* c = (gmiss_ctx*)c_;
    for (uint64_t i = b; i < e; ++i)
        c->out[i] = (uint8_t)grid_miss_one(c->coarse, c->CX, c->CY, c->CZ, c->shift, c->X, c->Y, c->Z, c->o + 3 * i, c->d + 3 * i);
}
void vo_grid_miss_test(const uint8_t* coarse, int CX, int CY, int CZ, int shift, int X, int Y, int Z, const float* origin,
                       const float* dir, uint64_t n, uint8_t* out, int threads) {
    gmiss_ctx c = {coarse, CX, CY, CZ, shift, X, Y, Z, origin, dir, out};
    par_for(gmiss_range, &c, n, 4096, threads);
}

/* ------------------------------------------------------------------------------------------ */
/* SVO<N>::castRay with the hit fill restored, include/svo.hpp:62-70,116-194; Ray volumetric.hpp:25-52 */
/* ------------------------------------------------------------------------------------------ */
typedef struct svo_ray {
    v3 start, dir, t, step, pos_dir;
    int side; float t_total;
    uint8_t** occ; int S;
    uint32_t max_iter;
    vo_hit* res;
} svo_ray;
static inline void clampf_(float* v, float lo, float hi) { if (*v > hi) *v = hi; else if (*v < lo) *v = lo; }   /* utils.cpp:67-75 */

/* node = cube of edge 2*cell_size whose low corner (voxel units) is (bx,by,bz); position is relative to it */
static void svo_rec(svo_ray* r, v3 position, uint32_t cell_size, int bx, int by, int bz) {
    const float cs = (float)cell_size;
    v3 ci = v3_((float)(int32_t)(position.x / cs), (float)(int32_t)(position.y / cs), (float)(int32_t)(position.z / cs));   /* :142 */
    clampf_(&ci.x, 0.0f, 1.0f); clampf_(&ci.y, 0.0f, 1.0f); clampf_(&ci.z, 0.0f, 1.0f);
    v3 tm = v3_(((ci.x + r->pos_dir.x) * cs - position.x) / r->dir.x,                                   /* :146 */
                ((ci.y + r->pos_dir.y) * cs - position.y) / r->dir.y,
                ((ci.z + r->pos_dir.z) * cs - position.z) / r->dir.z);
    const v3 t = v3_(cs * r->t.x, cs * r->t.y, cs * r->t.z);                                            /* :148 */
    float tmm = 0.0f;
    const float t_total = r->t_total;
    int l = 0;
    while ((1u << l) < cell_size) ++l;                 /* children are cubes of edge 2^l */
    const size_t n = (size_t)(r->S >> l);
    while (ci.x >= 0 && ci.y >= 0 && ci.z >= 0 && ci.x < 2 && ci.y < 2 && ci.z < 2 && r->res->complexity < r->max_iter) {   /* :152 */
        ++r->res->complexity;
        const int cx = bx + (int)(uint32_t)ci.x * (int)cell_size, cy = by + (int)(uint32_t)ci.y * (int)cell_size,
                  cz = bz + (int)(uint32_t)ci.z * (int)cell_size;
        if (r->occ[l][(((size_t)cx >> l) * n + ((size_t)cy >> l)) * n + ((size_t)cz >> l)]) {           /* :156-157 */
            if (cell_size == 1) {                                                                       /* leaf :158-161 */
                const float tt = t_total + tmm;
                vo_hit* h = r->res;
                const v3 hp = v3_(r->start.x + tt * r->dir.x, r->start.y + tt * r->dir.y, r->start.z + tt * r->dir.z);   /* :120 */
                h->hit = 1;
                h->position[0] = hp.x; h->position[1] = hp.y; h->position[2] = hp.z;
                h->distance = tt;
                if (r->side == 0) { h->normal[0] = -r->step.x; h->voxel_coord[0] = 1.0f - fracf_(hp.z); h->voxel_coord[1] = fracf_(hp.y); }
                else if (r->side == 1) { h->normal[1] = -r->step.y; h->voxel_coord[0] = fracf_(hp.x); h->voxel_coord[1] = fracf_(hp.z); }
                else { h->normal[2] = -r->step.z; h->voxel_coord[0] = fracf_(hp.x); h->voxel_coord[1] = fracf_(hp.y); }
                h->face = 1u << r->side;
                h->voxel[0] = cx; h->voxel[1] = cy; h->voxel[2] = cz;
                return;
            }
            const v3 sub = v3_((position.x + tmm * r->dir.x) - ci.x * cs,                               /* :164 */
                               (position.y + tmm * r->dir.y) - ci.y * cs,
                               (position.z + tmm * r->dir.z) - ci.z * cs);
            r->t_total = t_total + tmm;
            svo_rec(r, sub, cell_size >> 1, cx, cy, cz);
            if (r->res->hit) return;
        }
        if (tm.x < tm.y) {                                                                              /* :173-192 */
            if (tm.x < tm.z) { tmm = tm.x; tm.x += t.x; ci.x += r->step.x; r->side = 0; }
            else { tmm = tm.z; tm.z += t.z; ci.z += r->step.z; r->side = 2; }
        } else {
            if (tm.y < tm.z) { tmm = tm.y; tm.y += t.y; ci.y += r->step.y; r->side = 1; }
            else { tmm = tm.z; tm.z += t.z; ci.z += r->step.z; r->side = 2; }
        }
    }
}
typedef struct { uint8_t** occ; int depth; const float *o, *d; uint32_t max_iter; vo_hit* out; } svo_ctx;
static void svo_range(void* c_, uint64_t b, uint64_t e) {
    svo_ctx* c = (svo_ctx*)c_;
    for (uint64_t i = b; i < e; ++i) {
        vo_hit* res = c->out + i;
        memset(res, 0, sizeof(*res));
        svo_ray r;
        r.start = v3_(c->o[3 * i], c->o[3 * i + 1], c->o[3 * i + 2]);
        r.dir = v3_(c->d[3 * i], c->d[3 * i + 1], c->d[3 * i + 2]);
        r.t = v3_(fabsf(1.0f / r.dir.x), fabsf(1.0f / r.dir.y), fabsf(1.0f / r.dir.z));               /* volumetric.hpp:33 */
        r.step = v3_(r.dir.x >= 0.0f ? 1.0f : -1.0f, copysignf(1.0f, r.dir.y), copysignf(1.0f, r.dir.z));   /* :34 */
        r.pos_dir = v3_(r.dir.x > 0.0f, r.dir.y > 0.0f, r.dir.z > 0.0f);                               /* :35 */
        r.side = 0; r.t_total = 0.0f; r.occ = c->occ; r.S = 1 << c->depth; r.max_iter = c->max_iter; r.res = res;
        svo_rec(&r, r.start, 1u << (c->depth - 1), 0, 0, 0);                                            /* svo.hpp:66-67 */
    }
}
void vo_svo_cast(const uint8_t* occ, int depth, const float* origin, const float* dir, uint32_t max_iter, uint64_t n,
                 vo_hit* out, int threads) {
    svo_ctx c = {occ_pyramid(depth, occ), depth, origin, dir, max_iter, out};
    par_for(svo_range, &c, n, 4096, threads);
    occ_pyramid_free(c.occ, depth);
}

/* ------------------------------------------------------------------------------------------ */
/* RNG: Philox4x32-10 on the 100-level lattice of getRand (utils.cpp:77-81)                     */
/* ------------------------------------------------------------------------------------------ */
void vo_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
/* getRand(min,max) = min + (max-min) * (float(r % 100) / 100.0f), utils.cpp:77-81.
 * dimension d of sample s of pixel p: word (d & 3) of Philox(ctr = {p, s, d >> 2, 0}, key = seed). */
static float lattice_rand(const vo_render_params* p, uint32_t pixel, uint32_t sample, uint32_t dim, float lo, float hi) {
    const uint32_t ctr[4] = {pixel, sample, dim >> 2, 0u}, key[2] = {p->seed_lo, p->seed_hi};
    uint32_t w[4];
    vo_philox4x32_10(ctr, key, w);
    const float rv = (float)(w[dim & 3u] % 100u) / 100.0f;
    return lo + (hi - lo) * rv;
}

/* ------------------------------------------------------------------------------------------ */
/* Camera::getRay camera_controller.hpp:34-54 + lens mapping main.cpp:145-149                   */
/* ------------------------------------------------------------------------------------------ */
static inline v3 view_to_world(const float m[9], v3 v) {              /* v * rot_mat, :51-54 */
    return v3_(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z, m[6] * v.x + m[7] * v.y + m[8] * v.z);
}
void vo_camera_ray(const vo_render_params* p, int32_t x, int32_t y, int32_t sample, float origin[3], float dir[3]) {
    const float aspect = (float)p->width / (float)p->height;          /* main.cpp:133 */
    const float lens_x = (float)x / (float)p->height - aspect * 0.5f; /* main.cpp:145 */
    const float lens_y = (float)y / (float)p->height - 0.5f;          /* main.cpp:146 */
    const uint32_t pixel = (uint32_t)y * (uint32_t)p->width + (uint32_t)x;
    const float u0 = lattice_rand(p, pixel, (uint32_t)sample, 0, -0.5f, 0.5f);
    const float u1 = lattice_rand(p, pixel, (uint32_t)sample, 1, -0.5f, 0.5f);
    const v3 fn = norm3(v3_(lens_x, lens_y, p->fov));                 /* :37-39 */
    const v3 focal = v3_(fn.x * p->focal_length, fn.y * p->focal_length, fn.z * p->focal_length);
    const v3 rnd = v3_(p->aperture * u0, p->aperture * u1, p->aperture * 0.0f);   /* :40 */
    const v3 ray = norm3(v3_(focal.x - rnd.x, focal.y - rnd.y, focal.z - rnd.z)); /* :42 */
    const v3 wd = view_to_world(p->rot_mat, ray), wo = view_to_world(p->rot_mat, rnd);
    const float scale = 1.0f / (float)(1 << p->depth);                /* main.cpp:82 */
    origin[0] = (p->cam_position[0] + wo.x) * scale + 1.0f;           /* main.cpp:149 */
    origin[1] = (p->cam_position[1] + wo.y) * scale + 1.0f;
    origin[2] = (p->cam_position[2] + wo.z) * scale + 1.0f;
    dir[0] = wd.x; dir[1] = wd.y; dir[2] = wd.z;
}

/* ------------------------------------------------------------------------------------------ */
/* RayCaster::castRay / getGlobalIllumination / renderRay, include/raycaster.hpp:67-240         */
/* ------------------------------------------------------------------------------------------ */
typedef struct shade_ctx {
    const vo_lnode* nodes; const vo_render_params* p;
    const uint8_t *tex_top, *tex_side;
    uint32_t* accum; uint8_t* rgba;
    vo_render_stats* stats; pthread_mutex_t lock;
} shade_ctx;

static inline uint8_t mulc(uint8_t c, float f) { return (uint8_t)minf_(255.0f, (float)c * f); }   /* utils.cpp:43-48 */
static inline uint8_t addc(uint8_t a, uint8_t b) { int s = a + b; s = s < 255 ? s : 255; return (uint8_t)(s > 0 ? s : 0); }   /* :35-40 */

/* normalised GI estimate: sun_intensity * E is what raycaster.hpp:200-201 accumulates (bounces==1) */
static float gi_estimate(const shade_ctx* c, const vo_hit* pt, uint32_t pixel, uint32_t sample, int level, vo_render_stats* st) {
    const vo_render_params* p = c->p;
    const float n_norm = (1.0f / (float)(1 << p->depth)) * 0.0078125f * 2.0f;                      /* :171-172 */
    const v3 n = v3_(pt->normal[0], pt->normal[1], pt->normal[2]);
    const v3 start = v3_(pt->position[0] + n.x * n_norm, pt->position[1] + n.y * n_norm, pt->position[2] + n.z * n_norm);   /* :174 */
    const float c1 = lattice_rand(p, pixel, sample, 2u + 2u * (uint32_t)level, -1000.0f, 1000.0f);  /* :180-181 */
    const float c2 = lattice_rand(p, pixel, sample, 3u + 2u * (uint32_t)level, -1000.0f, 1000.0f);
    v3 noise;
    if (n.x != 0.0f) noise = v3_(0.0f, c1, c2);                                                    /* :182-190 */
    else if (n.y != 0.0f) noise = v3_(c1, 0.0f, c2);
    else if (n.z != 0.0f) noise = v3_(c1, c2, 0.0f);
    else return 0.0f;          /* noise_normal is uninitialised in the reference (start inside a solid) */
    const v3 gr = norm3(v3_((n.x + noise.x) * n_norm, (n.y + noise.y) * n_norm, (n.z + noise.z) * n_norm));   /* :192 */
    const float dot_gi = dot3(gr, n);                                                               /* :193 */
    vo_hit gp;
    const float so[3] = {start.x, start.y, start.z}, sd[3] = {gr.x, gr.y, gr.z};
    lsvo_cast_one(c->nodes, p->depth, p->guard, so, sd, 0.5f, 0.0f, &gp);                           /* :194 */
    st->rays[2 + 2 * level]++; st->complexity[2 + 2 * level] += gp.complexity;
    if (!gp.hit) return 0.0f;
    const v3 gn = v3_(gp.normal[0], gp.normal[1], gp.normal[2]);
    const v3 ls = v3_(gp.position[0] + gn.x * n_norm, gp.position[1] + gn.y * n_norm, gp.position[2] + gn.z * n_norm);   /* :196 */
    const v3 tl = norm3(v3_(p->light_position[0] - ls.x, p->light_position[1] - ls.y, p->light_position[2] - ls.z));    /* :197 */
    vo_hit lp;
    const float lo[3] = {ls.x, ls.y, ls.z}, ld[3] = {tl.x, tl.y, tl.z};
    lsvo_cast_one(c->nodes, p->depth, p->guard, lo, ld, 0.5f, 0.0f, &lp);                           /* :198 */
    st->rays[3 + 2 * level]++; st->complexity[3 + 2 * level] += lp.complexity;
    float irradiance = 0.0f;
    if (!lp.hit) irradiance = maxf_(0.0f, dot3(gn, tl));                                            /* :199-200 */
    if (level + 1 < p->gi_bounces) irradiance = irradiance + gi_estimate(c, &gp, pixel, sample, level + 1, st);   /* extension */
    return minf_(0.5f, irradiance * dot_gi);                                                        /* :201 */
}

static void shade_sample(const shade_ctx* c, int32_t x, int32_t y, int32_t sample, uint8_t rgb[3], vo_render_stats* st) {
    const vo_render_params* p = c->p;
    const uint32_t pixel = (uint32_t)y * (uint32_t)p->width + (uint32_t)x;
    float o[3], d[3];
    vo_camera_ray(p, x, y, sample, o, d);
    vo_hit h;
    const float SCALE = 1.0f / (float)(1 << p->depth);                                              /* :123-124 */
    rgb[0] = rgb[1] = rgb[2] = 0;                                                                   /* ColorResult: Black, :38 */
    /* Mirror reflections on LSVO frames — an EXTENSION ("parity unpinned": Cell::Mirror cell.hpp:8, RayContext::bounds and
     * max_bounds = 4 raycaster.hpp:13,127,277 exist, no code reflects).  The LSVO carries one shared Solid/Grass cell
     * (lsvo.hpp:21-23), so mirrors are given by a rule: with mirror_y1 > 0 the TOP faces (normal along y only) of the voxels
     * of layer y = mirror_y1 - 1 (castRay coordinates; the flat valley floors of the demo terrain are such a layer) are
     * Cell::Mirror.  A mirror hit with bounds < max_bounds continues from hit + normal * SCALE * 0.001 (the shadow-ray
     * offset of :139) with d.y negated, jittered by roughness * (r0, r1, r2) from dimensions 8+3b..10+3b of the sample's
     * Philox stream and re-normalised, tint *= 0.8 — the rule of vo_grid_render.  Reflection rays count as class 0. */
    float tint = 1.0f;
    int bounds = 0;
    for (;;) {
        lsvo_cast_one(c->nodes, p->depth, p->guard, o, d, 0.0f, 0.0f, &h);                          /* :131 */
        st->rays[0]++; st->complexity[0] += h.complexity;
        if (!h.hit) return;
        if (!(p->mirror_y1 > 0 && bounds < p->max_bounds && h.voxel[1] == p->mirror_y1 - 1 && h.normal[1] != 0.0f && h.normal[0] == 0.0f &&
              h.normal[2] == 0.0f))
            break;
        for (int a = 0; a < 3; ++a) o[a] = h.position[a] + h.normal[a] * SCALE * 0.001f;
        d[1] = -d[1];
        const float r0 = lattice_rand(p, pixel, (uint32_t)sample, 8u + 3u * (uint32_t)bounds, -0.5f, 0.5f);
        const float r1 = lattice_rand(p, pixel, (uint32_t)sample, 9u + 3u * (uint32_t)bounds, -0.5f, 0.5f);
        const float r2 = lattice_rand(p, pixel, (uint32_t)sample, 10u + 3u * (uint32_t)bounds, -0.5f, 0.5f);
        const v3 nd = norm3(v3_(d[0] + p->roughness * r0, d[1] + p->roughness * r1, d[2] + p->roughness * r2));
        d[0] = nd.x; d[1] = nd.y; d[2] = nd.z;
        tint = tint * 0.8f;
        ++bounds;
    }
    const v3 n = v3_(h.normal[0], h.normal[1], h.normal[2]);
    const v3 hp = v3_(h.position[0] + n.x * SCALE * 0.001f, h.position[1] + n.y * SCALE * 0.001f, h.position[2] + n.z * SCALE * 0.001f);   /* :139 */
    /* albedo: :141-145, :209-240 — the LSVO's single cell is Solid/Grass (lsvo.hpp:21-23) */
    const uint8_t* tex = n.y != 0.0f ? c->tex_top : c->tex_side;                                    /* :211-215 */
    float u = h.voxel_coord[0], v = h.voxel_coord[1];
    clampf_(&u, 0.0f, 1.0f); clampf_(&v, 0.0f, 1.0f);                                               /* :237-238 */
    const uint32_t tx = (uint32_t)(16.0f * u), ty = (uint32_t)(16.0f * v);                          /* :239 */
    const uint8_t* texel = tex + 3 * ((size_t)ty * 16 + tx);
    /* sun shadow: :147-159 (the 4 shadow samples of use_samples are identical rays → cast once) */
    const v3 tl = norm3(v3_(p->light_position[0] - hp.x, p->light_position[1] - hp.y, p->light_position[2] - hp.z));   /* :152 */
    vo_hit sh;
    const float so[3] = {hp.x, hp.y, hp.z}, sd[3] = {tl.x, tl.y, tl.z};
    lsvo_cast_one(c->nodes, p->depth, p->guard, so, sd, 0.0f, 0.0f, &sh);                           /* :153 */
    st->rays[1]++; st->complexity[1] += sh.complexity;
    float light = 0.0f;
    if (!sh.hit) light = maxf_(0.0f, dot3(tl, n));                                                  /* :155-157 */
    float gi = 0.0f;
    if (p->use_gi) gi = maxf_(0.0f, 1000000.0f * gi_estimate(c, &h, pixel, (uint32_t)sample, 0, st) / 1.0f);   /* :161, :201, :206 */
    const float f = minf_(1.0f, maxf_(0.0f, light + gi));                                           /* :163 */
    rgb[0] = mulc(mulc(texel[0], f), tint); rgb[1] = mulc(mulc(texel[1], f), tint); rgb[2] = mulc(mulc(texel[2], f), tint);   /* tint = 1: identity */
}

static void render_range(void* c_, uint64_t b, uint64_t e) {
    shade_ctx* c = (shade_ctx*)c_;
    const vo_render_params* p = c->p;
    vo_render_stats st; memset(&st, 0, sizeof(st));
    const uint64_t W = (uint64_t)p->width;
    for (uint64_t i = b; i < e; ++i) {
        const int32_t y = p->row_begin + (int32_t)(i / W), x = (int32_t)(i % W);
        if (p->tile_step > 1 && (((y - p->row_begin) >> 2) % p->tile_step) != p->tile_index) continue;
        if (p->checker) {                                                                           /* main.cpp:143 */
            const int32_t rel = p->checker_area_height > 0 ? y % p->checker_area_height : y;
            if ((rel & 1) != ((x + p->checker - 1) & 1)) continue;
        }
        const size_t px = (size_t)y * W + (size_t)x;
        for (int32_t s = 0; s < p->spp; ++s) {
            uint8_t rgb[3];
            shade_sample(c, x, y, p->sample_offset + s, rgb, &st);
            if (p->use_samples) {                                                                   /* :87-90 */
                if (c->accum) { uint32_t* a = c->accum + 4 * px; a[0] += rgb[0]; a[1] += rgb[1]; a[2] += rgb[2]; a[3] += 1u; }
            } else if (c->rgba) {                                                                   /* :79-85 */
                uint8_t* q = c->rgba + 4 * px;
                for (int k = 0; k < 3; ++k) q[k] = addc(mulc(q[k], 0.4f), mulc(rgb[k], 1.0f - 0.4f));
                q[3] = 255;
            }
        }
        if (p->use_samples && c->accum && c->rgba) {                                                /* :94-103 */
            const uint32_t* a = c->accum + 4 * px; uint8_t* q = c->rgba + 4 * px;
            for (int k = 0; k < 3; ++k) q[k] = (uint8_t)((double)a[k] / (double)a[3]);
            q[3] = 255;
        }
    }
    if (c->stats) {
        pthread_mutex_lock(&c->lock);
        for (int k = 0; k < 6; ++k) { c->stats->rays[k] += st.rays[k]; c->stats->complexity[k] += st.complexity[k]; }
        pthread_mutex_unlock(&c->lock);
    }
}

void vo_render(const vo_lnode* nodes, const vo_render_params* p, const uint8_t* tex_top, const uint8_t* tex_side,
               uint32_t* accum, uint8_t* rgba, vo_render_stats* stats) {
    shade_ctx c;
    c.nodes = nodes; c.p = p; c.tex_top = tex_top; c.tex_side = tex_side; c.accum = accum; c.rgba = rgba; c.stats = stats;
    pthread_mutex_init(&c.lock, NULL);
    if (stats) memset(stats, 0, sizeof(*stats));
    const int32_t r1 = p->row_end > p->row_begin ? p->row_end : p->height;
    const uint64_t n = (uint64_t)(r1 - p->row_begin) * (uint64_t)p->width;
    par_for(render_range, &c, n, 256, p->threads);
    pthread_mutex_destroy(&c.lock);
}

/* ------------------------------------------------------------------------------------------ */
/* Grid shading with mirror reflections — extension, specified in port.h / DESIGN.md §2         */
/* ------------------------------------------------------------------------------------------ */
typedef struct grid_shade_ctx {
    const uint8_t* cells; int X, Y, Z;
    const vo_render_params* p; const uint8_t *tex_top, *tex_side;
    uint32_t* accum; uint8_t* rgba; vo_render_stats* stats; pthread_mutex_t lock;
} grid_shade_ctx;

static void grid_shade_sample(const grid_shade_ctx* c, int32_t x, int32_t y, int32_t sample, uint8_t rgb[3], vo_render_stats* st) {
    const vo_render_params* p = c->p;
    const uint32_t pixel = (uint32_t)y * (uint32_t)p->width + (uint32_t)x;
    float o[3], d[3];
    {   /* Camera::getRay in voxel units */
        const float aspect = (float)p->width / (float)p->height;
        const float lens_x = (float)x / (float)p->height - aspect * 0.5f, lens_y = (float)y / (float)p->height - 0.5f;
        const float u0 = lattice_rand(p, pixel, (uint32_t)sample, 0, -0.5f, 0.5f), u1 = lattice_rand(p, pixel, (uint32_t)sample, 1, -0.5f, 0.5f);
        const v3 fn = norm3(v3_(lens_x, lens_y, p->fov));
        const v3 focal = v3_(fn.x * p->focal_length, fn.y * p->focal_length, fn.z * p->focal_length);
        const v3 rnd = v3_(p->aperture * u0, p->aperture * u1, p->aperture * 0.0f);
        const v3 ray = norm3(v3_(focal.x - rnd.x, focal.y - rnd.y, focal.z - rnd.z));
        const v3 wd = view_to_world(p->rot_mat, ray), wo = view_to_world(p->rot_mat, rnd);
        o[0] = p->cam_position[0] + wo.x; o[1] = p->cam_position[1] + wo.y; o[2] = p->cam_position[2] + wo.z;
        d[0] = wd.x; d[1] = wd.y; d[2] = wd.z;
    }
    rgb[0] = rgb[1] = rgb[2] = 0;
    float tint = 1.0f;
    int bounds = 0;
    for (;;) {
        vo_hit h; uint32_t steps;
        grid_cast_one(c->cells, c->X, c->Y, c->Z, o, d, &h, &steps);
        st->rays[bounds == 0 ? 0 : 2]++; st->complexity[bounds == 0 ? 0 : 2] += steps;
        if (!h.hit) return;
        const uint8_t type = c->cells[((size_t)h.voxel[0] * (size_t)c->Y + (size_t)h.voxel[1]) * (size_t)c->Z + (size_t)h.voxel[2]];
        const int axis = h.face == 1u ? 0 : (h.face == 2u ? 1 : 2);
        if (type == 2 && bounds < p->max_bounds) {                       /* Cell::Mirror */
            for (int a = 0; a < 3; ++a) o[a] = h.position[a] + h.normal[a] * 0.001f;
            d[axis] = -d[axis];
            const float r0 = lattice_rand(p, pixel, (uint32_t)sample, 8u + 3u * (uint32_t)bounds, -0.5f, 0.5f);
            const float r1 = lattice_rand(p, pixel, (uint32_t)sample, 9u + 3u * (uint32_t)bounds, -0.5f, 0.5f);
            const float r2 = lattice_rand(p, pixel, (uint32_t)sample, 10u + 3u * (uint32_t)bounds, -0.5f, 0.5f);
            const v3 nd = norm3(v3_(d[0] + p->roughness * r0, d[1] + p->roughness * r1, d[2] + p->roughness * r2));
            d[0] = nd.x; d[1] = nd.y; d[2] = nd.z;
            tint = tint * 0.8f;
            ++bounds;
            continue;
        }
        const uint8_t* tex = h.normal[1] != 0.0f ? c->tex_top : c->tex_side;
        float u = h.voxel_coord[0], v = h.voxel_coord[1];
        clampf_(&u, 0.0f, 1.0f); clampf_(&v, 0.0f, 1.0f);
        uint32_t tx = (uint32_t)(16.0f * u), ty = (uint32_t)(16.0f * v);
        if (tx > 15u) tx = 15u;                                          /* reference reads out of bounds at u == 1 (H6) */
        if (ty > 15u) ty = 15u;
        const uint8_t* texel = tex + 3 * ((size_t)ty * 16 + tx);
        float so[3], sd[3];
        for (int a = 0; a < 3; ++a) so[a] = h.position[a] + h.normal[a] * 0.001f;
        const v3 tl = norm3(v3_(p->light_position[0] - so[0], p->light_position[1] - so[1], p->light_position[2] - so[2]));
        sd[0] = tl.x; sd[1] = tl.y; sd[2] = tl.z;
        vo_hit sh; uint32_t ssteps;
        grid_cast_one(c->cells, c->X, c->Y, c->Z, so, sd, &sh, &ssteps);
        st->rays[1]++; st->complexity[1] += ssteps;
        float light = 0.0f;
        if (!sh.hit) light = maxf_(0.0f, dot3(tl, v3_(h.normal[0], h.normal[1], h.normal[2])));
        const float f = minf_(1.0f, maxf_(0.0f, light));
        for (int k = 0; k < 3; ++k) rgb[k] = mulc(mulc(texel[k], f), tint);
        return;
    }
}

static void grid_render_range(void* c_, uint64_t b, uint64_t e) {
    grid_shade_ctx* c = (grid_shade_ctx*)c_;
    const vo_render_params* p = c->p;
    vo_render_stats st; memset(&st, 0, sizeof(st));
    const uint64_t W = (uint64_t)p->width;
    for (uint64_t i = b; i < e; ++i) {
        const int32_t y = p->row_begin + (int32_t)(i / W), x = (int32_t)(i % W);
        if (p->tile_step > 1 && (((y - p->row_begin) >> 2) % p->tile_step) != p->tile_index) continue;
        if (p->checker) {                                                                           /* main.cpp:143, as vo_render */
            const int32_t rel = p->checker_area_height > 0 ? y % p->checker_area_height : y;
            if ((rel & 1) != ((x + p->checker - 1) & 1)) continue;
        }
        const size_t px = (size_t)y * W + (size_t)x;
        uint32_t* a = c->accum + 4 * px;
        for (int32_t s = 0; s < p->spp; ++s) {
            uint8_t rgb[3];
            grid_shade_sample(c, x, y, p->sample_offset + s, rgb, &st);
            a[0] += rgb[0]; a[1] += rgb[1]; a[2] += rgb[2]; a[3] += 1u;
        }
        if (c->rgba) {
            uint8_t* q = c->rgba + 4 * px;
            for (int k = 0; k < 3; ++k) q[k] = (uint8_t)((double)a[k] / (double)a[3]);
            q[3] = 255;
        }
    }
    if (c->stats) {
        pthread_mutex_lock(&c->lock);
        for (int k = 0; k < 6; ++k) { c->stats->rays[k] += st.rays[k]; c->stats->complexity[k] += st.complexity[k]; }
        pthread_mutex_unlock(&c->lock);
    }
}

void vo_grid_render(const uint8_t* cells, int X, int Y, int Z, const vo_render_params* p, const uint8_t* tex_top,
                    const uint8_t* tex_side, uint32_t* accum, uint8_t* rgba, vo_render_stats* stats) {
    grid_shade_ctx c;
    c.cells = cells; c.X = X; c.Y = Y; c.Z = Z; c.p = p; c.tex_top = tex_top; c.tex_side = tex_side;
    c.accum = accum; c.rgba = rgba; c.stats = stats;
    pthread_mutex_init(&c.lock, NULL);
    if (stats) memset(stats, 0, sizeof(*stats));
    const int32_t r1 = p->row_end > p->row_begin ? p->row_end : p->height;
    par_for(grid_render_range, &c, (uint64_t)(r1 - p->row_begin) * (uint64_t)p->width, 256, p->threads);
    pthread_mutex_destroy(&c.lock);
}

/* ------------------------------------------------------------------------------------------ */
/* Presentation: median + persistence blend, main.cpp:159-177 (specified in port.h)             */
static int cmp_u8_(const void* a, const void* b) { return (int)*(const uint8_t*)a - (int)*(const uint8_t*)b; }

void vo_present(const uint8_t* frame, uint8_t* display, int32_t width, int32_t height, int32_t median,
                float old_value_conservation) {
    const uint32_t c1 = (uint8_t)(255 * old_value_conservation);                 /* main.cpp:162 */
    const uint32_t c2 = (uint8_t)(255 * (1.0f - old_value_conservation));        /* main.cpp:164-165 */
    const int r = median == 3 ? 1 : median == 5 ? 2 : 0;
    for (int32_t y = 0; y < height; ++y)
        for (int32_t x = 0; x < width; ++x) {
            uint8_t* d = display + 4 * ((size_t)y * width + x);
            for (int k = 0; k < 3; ++k) {
                uint8_t w[25];
                int n = 0;
                for (int dy = -r; dy <= r; ++dy)
                    for (int dx = -r; dx <= r; ++dx) {
                        int sx = x + dx, sy = y + dy;
                        sx = sx < 0 ? 0 : sx >= width ? width - 1 : sx;
                        sy = sy < 0 ? 0 : sy >= height ? height - 1 : sy;
                        w[n++] = frame[4 * ((size_t)sy * width + sx) + k];
                    }
                qsort(w, (size_t)n, 1, cmp_u8_);
                const uint32_t f = w[n / 2];
                const uint32_t v = (d[k] * c1 + 127u) / 255u + (f * c2 + 127u) / 255u;
                d[k] = (uint8_t)(v > 255u ? 255u : v);
            }
            d[3] = 255;
        }
}
