/* TEST INFRASTRUCTURE ONLY: the CPU specification of point lights (DESIGN.md §2, "Point lights"), built on the CPU specification
 * of mirror voxels.  This file includes tests/cell_types_oracle.c (and through it tests/palette_oracle.c and oracle/port.c)
 * unchanged and adds
 *
 *   vo_render_point_lights(nodes, p, palette, types, lights, n_lights, tex_top, tex_side, accum, rgba, stats)
 *
 * which is vo_render_cell_types with one change: after the sun, each of the n_lights point lights {position, color, range}
 * (castRay frame, like light_position) adds its light to a per-channel sum L_c that starts at the sun term.  At the final
 * camera-chain hit, with n the raw normal and hp the sun shadow origin (raycaster.hpp:139), light i in index order:
 *
 *   v = P_i - hp;  dist = sqrtf((v.x*v.x + v.y*v.y) + v.z*v.z);  tl = norm3(v);  ndotl = dot3(tl, n)
 *   a shadow ray (origin hp, direction tl, coef 0) is cast iff dist < range_i && ndotl > 0   (counted as ray class 1)
 *   unless it hits at a distance < dist:  L_c = L_c + (color_i,c * ndotl) * (1.0f - dist / range_i)
 *
 * and then f_c = min(1, max(0, L_c + gi)), rgb_c = mult(mult(albedo_c, f_c), tint).  GI stays sun-only.  The two functions below
 * are cell_types_oracle.c's shade_sample_cell_types and render_range_cell_types with exactly that change;
 * tests/test_oracle_point_lights.py checks that no lights give vo_render_cell_types's frame.
 * Compiled by tests/point_lights_oracle.py with the oracle's flags. */
#include "cell_types_oracle.c"

/* vrt_point_light of include/vrt.h, 32 bytes */
typedef struct vo_point_light { float position[3]; float color[3]; float range; uint32_t reserved; } vo_point_light;

typedef struct point_lights_ctx {
    shade_ctx* shade; const uint8_t* palette; const uint8_t* types; const vo_point_light* lights; uint32_t n_lights;
} point_lights_ctx;

static void shade_sample_point_lights(const point_lights_ctx* lc, int32_t x, int32_t y, int32_t sample, uint8_t rgb[3],
                                      vo_render_stats* st) {
    const shade_ctx* c = lc->shade;
    const vo_render_params* p = c->p;
    const uint32_t pixel = (uint32_t)y * (uint32_t)p->width + (uint32_t)x;
    float o[3], d[3];
    vo_camera_ray(p, x, y, sample, o, d);
    vo_hit h;
    const float SCALE = 1.0f / (float)(1 << p->depth);                                              /* :123-124 */
    rgb[0] = rgb[1] = rgb[2] = 0;                                                                   /* ColorResult: Black, :38 */
    float tint = 1.0f;
    int bounds = 0;
    uint32_t leaf = 0u;
    for (;;) {
        lsvo_cast_leaf(c->nodes, p->depth, p->guard, o, d, 0.0f, 0.0f, &h, &leaf);                  /* :131 */
        st->rays[0]++; st->complexity[0] += h.complexity;
        if (!h.hit) return;
        const int lake = p->mirror_y1 > 0 && h.voxel[1] == p->mirror_y1 - 1 && h.normal[1] != 0.0f && h.normal[0] == 0.0f &&
                         h.normal[2] == 0.0f;
        int faces = 0, axis = 1;
        for (int a = 0; a < 3; ++a)
            if (h.normal[a] != 0.0f) { ++faces; axis = a; }
        const int typed = lc->types && lc->types[c->nodes[leaf].color] == 2 && faces == 1;
        if (!(bounds < p->max_bounds && (lake || typed))) break;
        for (int a = 0; a < 3; ++a) o[a] = h.position[a] + h.normal[a] * SCALE * 0.001f;
        d[axis] = -d[axis];
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
    const uint8_t* tex = n.y != 0.0f ? c->tex_top : c->tex_side;                                    /* :211-215 */
    float u = h.voxel_coord[0], v = h.voxel_coord[1];
    clampf_(&u, 0.0f, 1.0f); clampf_(&v, 0.0f, 1.0f);                                               /* :237-238 */
    const uint32_t tx = (uint32_t)(16.0f * u), ty = (uint32_t)(16.0f * v);                          /* :239 */
    const uint8_t* texel = tex + 3 * ((size_t)ty * 16 + tx);
    if (lc->palette) texel = lc->palette + 3 * (size_t)c->nodes[leaf].color;                        /* the final hit's colour */
    const v3 tl = norm3(v3_(p->light_position[0] - hp.x, p->light_position[1] - hp.y, p->light_position[2] - hp.z));   /* :152 */
    vo_hit sh;
    const float so[3] = {hp.x, hp.y, hp.z}, sd[3] = {tl.x, tl.y, tl.z};
    lsvo_cast_one(c->nodes, p->depth, p->guard, so, sd, 0.0f, 0.0f, &sh);                           /* :153 */
    st->rays[1]++; st->complexity[1] += sh.complexity;
    float light = 0.0f;
    if (!sh.hit) light = maxf_(0.0f, dot3(tl, n));                                                  /* :155-157 */
    /* point lights: per-channel sums that start at the sun term */
    float L[3] = {light, light, light};
    for (uint32_t i = 0; i < lc->n_lights; ++i) {
        const vo_point_light* pl = lc->lights + i;
        const v3 lv = v3_(pl->position[0] - hp.x, pl->position[1] - hp.y, pl->position[2] - hp.z);
        const float dist = sqrtf((lv.x * lv.x + lv.y * lv.y) + lv.z * lv.z);
        const v3 ld = norm3(lv);
        const float ndotl = dot3(ld, n);                                                            /* raw normal, as :156 */
        if (!(dist < pl->range && ndotl > 0.0f)) continue;       /* out of range, back-facing, zero normal, NaN: no ray */
        vo_hit lh;
        const float lo[3] = {hp.x, hp.y, hp.z}, ldir[3] = {ld.x, ld.y, ld.z};
        lsvo_cast_one(c->nodes, p->depth, p->guard, lo, ldir, 0.0f, 0.0f, &lh);
        st->rays[1]++; st->complexity[1] += lh.complexity;
        if (lh.hit && lh.distance < dist) continue;              /* a hit beyond the light does not shadow it */
        const float w = 1.0f - dist / pl->range;
        for (int k = 0; k < 3; ++k) L[k] = L[k] + (pl->color[k] * ndotl) * w;
    }
    float gi = 0.0f;
    if (p->use_gi) gi = maxf_(0.0f, 1000000.0f * gi_estimate(c, &h, pixel, (uint32_t)sample, 0, st) / 1.0f);   /* :161, :201, :206 */
    for (int k = 0; k < 3; ++k) {
        const float f = minf_(1.0f, maxf_(0.0f, L[k] + gi));                                        /* :163 per channel */
        rgb[k] = mulc(mulc(texel[k], f), tint);
    }
}

static void render_range_point_lights(void* c_, uint64_t b, uint64_t e) {
    const point_lights_ctx* lc = (const point_lights_ctx*)c_;
    shade_ctx* c = lc->shade;
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
            shade_sample_point_lights(lc, x, y, p->sample_offset + s, rgb, &st);
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

void vo_render_point_lights(const vo_lnode* nodes, const vo_render_params* p, const uint8_t* palette, const uint8_t* types,
                            const vo_point_light* lights, uint32_t n_lights, const uint8_t* tex_top, const uint8_t* tex_side,
                            uint32_t* accum, uint8_t* rgba, vo_render_stats* stats) {
    shade_ctx c;
    c.nodes = nodes; c.p = p; c.tex_top = tex_top; c.tex_side = tex_side; c.accum = accum; c.rgba = rgba; c.stats = stats;
    pthread_mutex_init(&c.lock, NULL);
    if (stats) memset(stats, 0, sizeof(*stats));
    point_lights_ctx lc = {&c, palette, types, lights, lights ? n_lights : 0u};
    const int32_t r1 = p->row_end > p->row_begin ? p->row_end : p->height;
    const uint64_t n = (uint64_t)(r1 - p->row_begin) * (uint64_t)p->width;
    par_for(render_range_point_lights, &lc, n, 256, p->threads);
    pthread_mutex_destroy(&c.lock);
}
