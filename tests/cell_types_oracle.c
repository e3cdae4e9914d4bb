/* TEST INFRASTRUCTURE ONLY: the CPU specification of mirror voxels (DESIGN.md §2, "Mirror voxels"), built on the CPU
 * specification of per-voxel colours.  This file includes tests/palette_oracle.c (and through it oracle/port.c) unchanged and adds
 *
 *   vo_render_cell_types(nodes, p, palette, types, tex_top, tex_side, accum, rgba, stats)
 *
 * which is vo_render_palette with one change: a table types[256] (NULL = all Solid) gives the Cell::Type of the voxels of each
 * colour, 1 = Solid, 2 = Mirror.  A hit of a camera-chain ray (the camera ray or a reflected one) on a voxel whose colour c (the
 * `color` byte of the leaf slot the walk ended in, as palette frames read it) has types[c] == Mirror reflects when
 * bounds < max_bounds and the raw normal has exactly one non-zero component a: the lake rule's reflection with d[a] negated
 * instead of d.y.  A hit reflects once if either rule holds.  Zero normals and edge or corner hits, sun-shadow and GI rays are
 * unchanged.  The two functions below are palette_oracle.c's shade_sample_palette and render_range_palette with exactly that
 * change; tests/test_oracle_cell_types.py checks that an all-Solid table gives vo_render_palette's frame.
 * Compiled by tests/cell_types_oracle.py with the oracle's flags. */
#include "palette_oracle.c"

typedef struct cell_types_ctx { shade_ctx* shade; const uint8_t* palette; const uint8_t* types; } cell_types_ctx;

static void shade_sample_cell_types(const shade_ctx* c, const uint8_t* palette, const uint8_t* types, int32_t x, int32_t y,
                                    int32_t sample, uint8_t rgb[3], vo_render_stats* st) {
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
        /* the lake: top faces of layer mirror_y1 - 1 (shade_sample_palette) */
        const int lake = p->mirror_y1 > 0 && h.voxel[1] == p->mirror_y1 - 1 && h.normal[1] != 0.0f && h.normal[0] == 0.0f &&
                         h.normal[2] == 0.0f;
        /* mirror voxels: the colour of the leaf slot the walk ended in, and the one axis of the face it hit */
        int faces = 0, axis = 1;
        for (int a = 0; a < 3; ++a)
            if (h.normal[a] != 0.0f) { ++faces; axis = a; }
        const int typed = types && types[c->nodes[leaf].color] == 2 && faces == 1;
        if (!(bounds < p->max_bounds && (lake || typed))) break;
        for (int a = 0; a < 3; ++a) o[a] = h.position[a] + h.normal[a] * SCALE * 0.001f;
        d[axis] = -d[axis];                                                                         /* the lake: axis = y */
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
    if (palette) texel = palette + 3 * (size_t)c->nodes[leaf].color;                                /* the final hit's colour */
    const v3 tl = norm3(v3_(p->light_position[0] - hp.x, p->light_position[1] - hp.y, p->light_position[2] - hp.z));   /* :152 */
    vo_hit sh;
    const float so[3] = {hp.x, hp.y, hp.z}, sd[3] = {tl.x, tl.y, tl.z};
    lsvo_cast_one(c->nodes, p->depth, p->guard, so, sd, 0.0f, 0.0f, &sh);                           /* :153: mirrors are solids */
    st->rays[1]++; st->complexity[1] += sh.complexity;
    float light = 0.0f;
    if (!sh.hit) light = maxf_(0.0f, dot3(tl, n));                                                  /* :155-157 */
    float gi = 0.0f;
    if (p->use_gi) gi = maxf_(0.0f, 1000000.0f * gi_estimate(c, &h, pixel, (uint32_t)sample, 0, st) / 1.0f);   /* :161, :201, :206 */
    const float f = minf_(1.0f, maxf_(0.0f, light + gi));                                           /* :163 */
    rgb[0] = mulc(mulc(texel[0], f), tint); rgb[1] = mulc(mulc(texel[1], f), tint); rgb[2] = mulc(mulc(texel[2], f), tint);
}

static void render_range_cell_types(void* c_, uint64_t b, uint64_t e) {
    const cell_types_ctx* tc = (const cell_types_ctx*)c_;
    shade_ctx* c = tc->shade;
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
            shade_sample_cell_types(c, tc->palette, tc->types, x, y, p->sample_offset + s, rgb, &st);
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

void vo_render_cell_types(const vo_lnode* nodes, const vo_render_params* p, const uint8_t* palette, const uint8_t* types,
                          const uint8_t* tex_top, const uint8_t* tex_side, uint32_t* accum, uint8_t* rgba, vo_render_stats* stats) {
    shade_ctx c;
    c.nodes = nodes; c.p = p; c.tex_top = tex_top; c.tex_side = tex_side; c.accum = accum; c.rgba = rgba; c.stats = stats;
    pthread_mutex_init(&c.lock, NULL);
    if (stats) memset(stats, 0, sizeof(*stats));
    cell_types_ctx tc = {&c, palette, types};
    const int32_t r1 = p->row_end > p->row_begin ? p->row_end : p->height;
    const uint64_t n = (uint64_t)(r1 - p->row_begin) * (uint64_t)p->width;
    par_for(render_range_cell_types, &tc, n, 256, p->threads);
    pthread_mutex_destroy(&c.lock);
}
