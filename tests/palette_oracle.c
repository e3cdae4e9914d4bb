/* TEST INFRASTRUCTURE ONLY: the CPU specification of per-voxel colours (DESIGN.md §2, "Per-voxel colours"), built on the
 * oracle's own restatement.  This file includes oracle/port.c and adds
 *
 *   vo_render_palette(nodes, p, palette, tex_top, tex_side, accum, rgba, stats)
 *
 * which is vo_render with one change: with a palette (256 RGB entries, or NULL = the textures), a sample's albedo is
 * palette[c] instead of the texel, c = the `color` byte of the leaf slot of the voxel its camera ray hits (after mirror bounces,
 * the last hit).  The slot is taken from the walk itself, nodes[N + child_offset + s] for the node N and child s at its leaf exit
 * (lsvo.hpp:90-95): independent of the device, which descends the array from the hit cell's coordinates.  Shadows, GI, the
 * mirror tint and the mult rounding are vo_render's.  The three functions below are port.c's lsvo_cast_one, shade_sample and
 * render_range with exactly those changes; tests/test_oracle_palette.py checks that a NULL palette gives vo_render's frame.
 * Compiled by tests/palette_oracle.py with the oracle's flags. */
#include "port.c"

typedef struct palette_ctx { shade_ctx* shade; const uint8_t* palette; } palette_ctx;

static void lsvo_cast_leaf(const vo_lnode* nodes, int depth, int guard, const float o[3], const float din[3],
                           float coef, float bias, vo_hit* res, uint32_t* leaf_slot) {
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
                if ((nd.leaf_mask >> shift) & 1u) {                   /* :90-95 */
                    *leaf_slot = parent + nd.child_offset + shift;    /* the hit voxel's own slot */
                    hit = 1;
                    break;
                }
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

static void shade_sample_palette(const shade_ctx* c, const uint8_t* palette, int32_t x, int32_t y, int32_t sample, uint8_t rgb[3], vo_render_stats* st) {
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
    uint32_t leaf = 0u;
    for (;;) {
        lsvo_cast_leaf(c->nodes, p->depth, p->guard, o, d, 0.0f, 0.0f, &h, &leaf);                  /* :131 */
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
    /* the palette replaces the texel: entry `color` of the leaf slot the walk above ended in (a camera ray has no cone, so
     * every hit is a leaf exit) */
    if (palette) texel = palette + 3 * (size_t)c->nodes[leaf].color;
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

static void render_range_palette(void* c_, uint64_t b, uint64_t e) {
    const palette_ctx* pc = (const palette_ctx*)c_;
    shade_ctx* c = pc->shade;
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
            shade_sample_palette(c, pc->palette, x, y, p->sample_offset + s, rgb, &st);
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

void vo_render_palette(const vo_lnode* nodes, const vo_render_params* p, const uint8_t* palette, const uint8_t* tex_top,
                       const uint8_t* tex_side, uint32_t* accum, uint8_t* rgba, vo_render_stats* stats) {
    shade_ctx c;
    c.nodes = nodes; c.p = p; c.tex_top = tex_top; c.tex_side = tex_side; c.accum = accum; c.rgba = rgba; c.stats = stats;
    pthread_mutex_init(&c.lock, NULL);
    if (stats) memset(stats, 0, sizeof(*stats));
    palette_ctx pc = {&c, palette};
    const int32_t r1 = p->row_end > p->row_begin ? p->row_end : p->height;
    const uint64_t n = (uint64_t)(r1 - p->row_begin) * (uint64_t)p->width;
    par_for(render_range_palette, &pc, n, 256, p->threads);
    pthread_mutex_destroy(&c.lock);
}
