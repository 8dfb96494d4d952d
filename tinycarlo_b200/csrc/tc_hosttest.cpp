// tc_hosttest.cpp — CPU-only TEST build of the kernel arithmetic (tc_core.cuh) with one lane per group.
//
// NOT part of the product: nothing under tinycarlo_b200/*.py loads this library. It exists so that the
// node-parallel clip passes, the closed-form rasteriser and the tracking logic that the CUDA kernels run can be
// checked against the oracle in a container without a GPU (tests/test_core_host.py), and the blob noise against cv2
// (tests/test_noise_host.py). The glue below mirrors the
// kernels in tc_kernels.cuh step by step (same pass order, same ping-pong flags), sequentially.
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "tc_core.cuh"
#include "tc_cull.h"
#include "tc_pack.h"
#include "tc_route.h"

#define HT_API extern "C" __attribute__((visibility("default")))

struct HtMap {
    TcPacked pk;
    TcNear near;   // nearest-laneline index, as tc_create builds it
    std::vector<TcClassTables> cls;
    std::vector<int32_t> edge_off;
    int C, sumE;
    uint8_t colors[TC_MAX_CLASSES * 3];
};

HT_API HtMap *ht_map_create(const TcMapDesc *map) {
    HtMap *m = new HtMap();
    std::string err = tc_pack_map(map, m->pk);
    if (!err.empty()) { delete m; return nullptr; }
    tc_class_views(map, m->pk, m->pk.blob.data(), m->pk.adj.data(), m->cls);
    m->C = map->n_classes;
    m->sumE = map->ll_edge_off[m->C];
    m->edge_off.assign(map->ll_edge_off, map->ll_edge_off + m->C + 1);
    memcpy(m->colors, map->ll_colors, (size_t)3 * m->C);
    tc_build_near(map, 1.0, 16384, m->near);
    return m;
}
HT_API void ht_map_destroy(HtMap *m) { delete m; }

static void ht_attach_near(const HtMap *m, TcTrackTables &t, bool use) {
    if (!use || m->near.nx == 0) return;
    t.near_x0 = m->near.x0; t.near_y0 = m->near.y0; t.near_inv_cell = m->near.inv_cell; t.near_nx = m->near.nx; t.near_ny = m->near.ny;
    t.near_off = m->near.off.data(); t.near_edge = m->near.edge.data();
}

// mirrors tc_track_kernel for n envs (mode 0 step / 1 reset) with n_cams cameras each: cam / pose are per view
// v = env * n_cams + m; view_mask (optional, reset with a mask) receives mask[env] for each view, as the kernels write it
HT_API void ht_track_rig(const HtMap *m, int n, int n_cams, int mode, int wrapped, double *sf, int32_t *si, const double *car, const double *cam,
                         double *pose, const float *act_cc, const int32_t *act_man, const uint8_t *mask, const int32_t *spawn,
                         double *info_f64, int32_t *nearest, uint8_t *terminated, uint8_t *truncated, uint8_t *view_mask) {
    TcTrackTables t = tc_track_tables(m->pk.blob.data(), m->pk.L);
    ht_attach_near(m, t, true);
    TcLanes g = {0, 1};
    const int C = m->C;
    for (int env = 0; env < n; env++) {
        const double *cp = car + (size_t)env * TC_CP_N;
        TcCarState s;
        bool trunc = false;
        if (mode == 1) {
            if (view_mask && mask) for (int k = 0; k < n_cams; k++) view_mask[(size_t)env * n_cams + k] = mask[env];
            if (mask && !mask[env]) continue;
            tc_load_state(sf + (size_t)env * TC_SF_N, si + (size_t)env * TC_SI_N, s);
            if (!tc_car_reset(t, cp, s, spawn[env])) continue;
        } else {
            tc_load_state(sf + (size_t)env * TC_SF_N, si + (size_t)env * TC_SI_N, s);
            double v = tc_np_clip((double)act_cc[2 * env], -1.0, 1.0), st = tc_np_clip((double)act_cc[2 * env + 1], -1.0, 1.0);
            trunc = tc_car_step(g, t, cp, s, v, st, act_man[env]);
        }
        double dist[TC_MAX_CLASSES];
        int near[TC_MAX_CLASSES];
        TcInfo info = tc_get_info(g, t, cp, s, wrapped != 0, dist, near);
        tc_store_state(sf + (size_t)env * TC_SF_N, si + (size_t)env * TC_SI_N, s);
        const double c = cos(s.rot), sn = sin(s.rot);
        for (int k = 0; k < n_cams; k++) {
            const size_t v = (size_t)env * n_cams + k;
            tc_camera_pose(cam + v * TC_CAM_N + TC_CAM_E, s.x, s.y, c, sn, pose + v * 12);
        }
        double *r = info_f64 + (size_t)env * (4 + C);
        r[0] = info.cte; r[1] = info.heading; r[2] = info.velocity;
        if (mode == 0) r[3] = info.reward;
        for (int c = 0; c < C; c++) { r[4 + c] = dist[c]; nearest[(size_t)env * C + c] = near[c]; }
        if (mode == 0) { terminated[env] = info.terminated; truncated[env] = trunc; }
    }
}
HT_API void ht_track(const HtMap *m, int n, int mode, int wrapped, double *sf, int32_t *si, const double *car, const double *cam,
                     double *pose, const float *act_cc, const int32_t *act_man, const uint8_t *mask, const int32_t *spawn,
                     double *info_f64, int32_t *nearest, uint8_t *terminated, uint8_t *truncated) {
    ht_track_rig(m, n, 1, mode, wrapped, sf, si, car, cam, pose, act_cc, act_man, mask, spawn, info_f64, nearest, terminated, truncated, nullptr);
}

// mirrors tc_project_kernel for one (env, class)
static int ht_project_one(const TcClassTables &ct, const double *pose, const double *cam, int H, int W, int32_t *seg) {
    int n = ct.n_nodes, m = ct.n_edges;
    std::vector<double> Px(n + 1), Py(n + 1), Pz(n + 1);
    std::vector<int32_t> ix(n + 1), iy(n + 1);
    std::vector<uint8_t> fA(n + 1), fB(n + 1), rA(n + 1), rB(n + 1), vis(n + 1);
    TcProjScratch sc = {Px.data(), Py.data(), Pz.data(), ix.data(), iy.data(), fA.data(), rA.data(), vis.data()};
    double max_range = cam[TC_CAM_MAX_RANGE];
    for (int v = 0; v < n; v++) {
        tc_transform_node(pose, ct.nodes[2 * v], ct.nodes[2 * v + 1], Px[v], Py[v], Pz[v]);
        fA[v] = Pz[v] < 0;
    }
    for (int v = 0; v < n; v++) fB[v] = fA[v] | (uint8_t)tc_clip_pass_node(ct, sc, fA.data(), v, true, -0.0000001);
    for (int v = 0; v < n; v++) fA[v] = fB[v] | (uint8_t)tc_clip_pass_node(ct, sc, fB.data(), v, false, -0.0000001);
    for (int v = 0; v < n; v++) rA[v] = Pz[v] > -max_range;
    for (int v = 0; v < n; v++) rB[v] = rA[v] | (uint8_t)tc_clip_pass_node(ct, sc, rA.data(), v, true, -max_range);
    for (int v = 0; v < n; v++) rA[v] = rB[v] | (uint8_t)tc_clip_pass_node(ct, sc, rB.data(), v, false, -max_range);
    for (int v = 0; v < n; v++) {
        double u, w;
        tc_project(cam, Px[v], Py[v], Pz[v], u, w);
        ix[v] = tc_np_int32(u);
        iy[v] = tc_np_int32(w);
        vis[v] = (u > 0 && u < W && w > 0 && w < H && fA[v] && rA[v]) ? 1 : 0;
    }
    int cnt = 0;
    for (int e = 0; e < m; e++) {
        int n0 = ct.edges[2 * e], n1 = ct.edges[2 * e + 1];
        if (!(vis[n0] || vis[n1])) continue;
        seg[4 * cnt] = ix[n0]; seg[4 * cnt + 1] = iy[n0]; seg[4 * cnt + 2] = ix[n1]; seg[4 * cnt + 3] = iy[n1];
        cnt++;
    }
    return cnt;
}

// mirrors tc_project_kernel + tc_raster_*_kernel (bands included) for n envs
HT_API void ht_render(const HtMap *m, int n, int H, int W, int fmt, int rows_per_band, const double *pose, const double *cam,
                      const int32_t *thickness, const uint8_t *mask, uint8_t *obs, int32_t *seg_count, int32_t *seg) {
    const int C = m->C;
    TcLanes g = {0, 1};
    if (rows_per_band <= 0) rows_per_band = H;
    const int n_bands = (H + rows_per_band - 1) / rows_per_band;
    const int plane_words = (int)(((size_t)rows_per_band * W + 31) / 32) + 1;
    for (int env = 0; env < n; env++) {
        if (mask && !mask[env]) continue;
        for (int c = 0; c < C; c++)
            seg_count[(size_t)env * C + c] = ht_project_one(m->cls[c], pose + (size_t)env * 12, cam + (size_t)env * TC_CAM_N, H, W,
                                                            seg + ((size_t)env * m->sumE + m->edge_off[c]) * 4);
        if (!obs) continue;
        for (int band = 0; band < n_bands; band++) {
            int y_lo = band * rows_per_band, y_hi = y_lo + rows_per_band < H ? y_lo + rows_per_band : H;
            std::vector<uint32_t> planes((size_t)C * plane_words, 0);
            for (int c = 0; c < C; c++) {
                TcPlane pl = {planes.data() + (size_t)c * plane_words, H, W, y_lo, y_hi, y_lo};
                const int32_t *s = seg + ((size_t)env * m->sumE + m->edge_off[c]) * 4;
                for (int k = 0; k < seg_count[(size_t)env * C + c]; k++) tc_polyline2(g, pl, s[4 * k], s[4 * k + 1], s[4 * k + 2], s[4 * k + 3], thickness[env]);
            }
            size_t npx = (size_t)(y_hi - y_lo) * W;
            for (size_t p = 0; p < npx; p++) {
                if (fmt == TC_OBS_CLASSES) {
                    for (int c = 0; c < C; c++)
                        obs[(((size_t)env * C + c) * H + y_lo) * W + p] = ((planes[(size_t)c * plane_words + (p >> 5)] >> (p & 31)) & 1) ? 255 : 0;
                } else {
                    uint8_t *o = obs + (((size_t)env * H + y_lo) * W + p) * 3;
                    o[0] = o[1] = o[2] = 0;
                    for (int c = 0; c < C; c++)
                        if ((planes[(size_t)c * plane_words + (p >> 5)] >> (p & 31)) & 1) memcpy(o, m->colors + 3 * c, 3);
                }
            }
        }
    }
}

// one polyline into a byte image through the bit-plane rasteriser (fuzzed against cv2 / the oracle)
// nlanes > 1 replays the work split of a warp lane by lane (lanes only interact through ORs into the plane)
HT_API void ht_polyline(uint8_t *img, int H, int W, int32_t x0, int32_t y0, int32_t x1, int32_t y1, int thickness, int y_lo, int y_hi,
                        int nlanes) {
    if (y_hi <= 0) { y_lo = 0; y_hi = H; }
    if (nlanes == 0) nlanes = 1;
    std::vector<uint32_t> plane(((size_t)(y_hi - y_lo) * W + 31) / 32 + 1, 0);
    TcPlane pl = {plane.data(), H, W, y_lo, y_hi, y_lo};
    if (nlanes < 0) {
        // the fused kernel's split: every role sets up its own slots (as different warps do), then 32 lanes draw
        TcPrim prims[TC_MAX_PRIMS_PER_SEG];
        for (int i = 0; i < TC_MAX_PRIMS_PER_SEG; i++) prims[i].kind = TC_PRIM_NONE;
        // nlanes == -2: the block-per-env kernels' set-up variant (one code instance for the edge roles, walker slopes up front)
        for (int role = 0; role < TC_N_ROLES; role++) {
            if (nlanes == -2) tc_polyline_setup<true>(W, H, x0, y0, x1, y1, thickness, role, prims);
            else tc_polyline_setup(W, H, x0, y0, x1, y1, thickness, role, prims);
        }
        for (int lane = 0; lane < 32; lane++) {
            TcLanes g = {lane, 32};
            for (int i = 0; i < TC_MAX_PRIMS_PER_SEG; i++)
                if (prims[i].kind != TC_PRIM_NONE) tc_prim_draw(g, pl, prims[i]);
        }
    } else
    for (int lane = 0; lane < nlanes; lane++) {
        TcLanes g = {lane, nlanes};
        tc_polyline2(g, pl, x0, y0, x1, y1, thickness);
    }
    for (size_t p = 0; p < (size_t)(y_hi - y_lo) * W; p++)
        if ((plane[p >> 5] >> (p & 31)) & 1) img[(size_t)y_lo * W + p] = 255;
}

// mirrors tc_bev_kernel for n envs at state rows sf [n,TC_SF_N] / si [n,TC_SI_N] (the route planes read the local path from
// si); out: u8 [n,P,H,W] 0/255, P = C + route (cos / sin are the host libm's)
HT_API void ht_bev(const HtMap *m, int n, const double *sf, const int32_t *si, const TcBevDesc *d, uint8_t *out) {
    const TcTrackTables tt = tc_track_tables(m->pk.blob.data(), m->pk.L);
    const TcBevGeom g = {d->pixel_per_meter, d->car_col, d->car_row, d->height, d->width, d->line_thickness, d->route};
    const int P = m->C + (d->route ? 1 : 0), H = d->height, W = d->width;
    const size_t npx = (size_t)P * H * W;
    const TcLanes lanes = {0, 1};
    for (int env = 0; env < n; env++) {
        const double *s = sf + (size_t)env * TC_SF_N;
        const int32_t *r = si + (size_t)env * TC_SI_N;
        const double c = cos(s[TC_SF_ROT]), sn = sin(s[TC_SF_ROT]);
        std::vector<uint32_t> plane(npx / 32 + 2, 0);
        for (int i = 0; i < m->sumE + 4; i++) {
            int32_t p[4];
            int q = 0;
            if (!tc_bev_segment(tt, g, s[TC_SF_X], s[TC_SF_Y], c, sn, r, i, p, q)) continue;
            const TcPlane pl = {plane.data(), H, W, 0, H, -q * H};
            tc_polyline2(lanes, pl, p[0], p[1], p[2], p[3], g.thickness);
        }
        for (size_t b = 0; b < npx; b++) out[(size_t)env * npx + b] = ((plane[b >> 5] >> (b & 31)) & 1) ? 255 : 0;
    }
}

// mirrors tc_lidar_kernel for n envs at state rows sf [n,TC_SF_N]: out_f64 [n,C,R] is the scan in float64, before the float32
// cast (cos / sin of the heading and of the ray angles are the host libm's, as tc_set_lidar computes the latter)
HT_API void ht_lidar(const HtMap *m, int n, const double *sf, const TcLidarDesc *d, double *out_f64) {
    const TcTrackTables tt = tc_track_tables(m->pk.blob.data(), m->pk.L);
    const TcLidarGeom g = {d->rays, d->fov, d->max_range, d->origin_forward, d->origin_right};
    const int C = m->C, R = d->rays;
    std::vector<double> a(R), b(R), best(R);
    for (int j = 0; j < R; j++) {
        const double phi = (d->fov * ((j + 0.5) / R) - d->fov / 2) * (TC_PI / 180.0);
        a[j] = cos(phi);
        b[j] = sin(phi);
    }
    for (int env = 0; env < n; env++) {
        const double *s = sf + (size_t)env * TC_SF_N;
        const double c = cos(s[TC_SF_ROT]), sn = sin(s[TC_SF_ROT]);
        double ox, oy;
        tc_lidar_origin(g, s[TC_SF_X], s[TC_SF_Y], c, sn, ox, oy);
        for (int p = 0; p < C; p++) {
            const double *nodes = tt.ll_nodes + 2 * tt.ll_node_off[p];
            for (int j = 0; j < R; j++) best[j] = g.max_range;
            for (int i = tt.ll_edge_off[p]; i < tt.ll_edge_off[p + 1]; i++) {
                const int32_t n0 = tt.ll_edges[2 * i], n1 = tt.ll_edges[2 * i + 1];
                double st[5];
                if (!tc_lidar_stage(g, ox, oy, c, sn, nodes[2 * n0], nodes[2 * n0 + 1], nodes[2 * n1], nodes[2 * n1 + 1], st)) continue;
                for (int j = 0; j < R; j++) {
                    double dx, dy, t;
                    tc_lidar_dir(a[j], b[j], c, sn, dx, dy);
                    if (tc_lidar_hit(dx, dy, st[0], st[1], st[2], st[3], st[4], t) && t < best[j]) best[j] = t;
                }
            }
            double *o = out_f64 + ((size_t)env * C + p) * R;
            for (int j = 0; j < R; j++) o[j] = best[j] == 0 ? 0.0 : best[j];
        }
    }
}

// the cull of the scan (tc_lidar_stage) for one edge: 1 kept, 0 dropped
HT_API int ht_lidar_keep(const TcLidarDesc *d, double ox, double oy, double c, double s, double ax, double ay, double bx, double by) {
    const TcLidarGeom g = {d->rays, d->fov, d->max_range, d->origin_forward, d->origin_right};
    double st[5];
    return tc_lidar_stage(g, ox, oy, c, s, ax, ay, bx, by, st) ? 1 : 0;
}

// the route table of tc_set_route (tc_route.h) for goals[0..G-1]: D [G][Q], cmd [G][Q]
HT_API void ht_route_table(const HtMap *m, int G, const int32_t *goals, double *D, int8_t *cmd) {
    tc_build_route(tc_track_tables(m->pk.blob.data(), m->pk.L), goals, G, D, cmd);
}

// mirrors tc_route_kernel for n envs at states sf / si (mode, mask, was_reset as there; terminated / done optional, OR-ed)
HT_API void ht_route_update(const HtMap *m, int G, const int32_t *goals, const double *D, const int8_t *cmd, double reach, int on_reach,
                            int n, int mode, const double *sf, const int32_t *si, const uint8_t *mask, const uint8_t *was_reset,
                            uint64_t *rng, int32_t *goal_index, double *prev, int32_t *goal, float *goal_position, int32_t *command,
                            float *distance, float *progress, uint8_t *reached, uint8_t *terminated, uint8_t *done) {
    const TcTrackTables t = tc_track_tables(m->pk.blob.data(), m->pk.L);
    TcRoute r;
    r.D = D; r.cmd = cmd; r.goals = goals; r.G = G; r.Q = t.lp_n_edges; r.reach = reach; r.on_reach = on_reach;
    TcRouteOutputs o = {goal, goal_position, command, distance, progress, reached};
    for (int i = 0; i < n; i++) {
        if (mode != 0 && mask && !mask[i]) continue;
        const double *s = sf + (size_t)i * TC_SF_N;
        int32_t k = goal_index[i];
        double p = prev[i], dist, prog;
        int c;
        bool re, term;
        tc_route_update(t, r, mode, was_reset && was_reset[i], si + (size_t)i * TC_SI_N, s[TC_SF_FRONT_X], s[TC_SF_FRONT_Y],
                        rng + (size_t)i * TC_RNG_N, k, p, c, dist, prog, re, term);
        goal_index[i] = k;
        prev[i] = p;
        tc_route_store(t, r, o, i, k, c, dist, prog, re);
        if (term) {
            if (terminated) terminated[i] = 1;
            if (done) done[i] = 1;
        }
    }
}

// the reset paths' spawn draws (tc_spawn_draw): k consecutive draws of n env streams, states advanced in place
HT_API void ht_spawn_draws(const HtMap *m, int n, uint64_t *rng_state, const int32_t *spawn_points, int n_spawn_points, int k, int32_t *out) {
    TcTrackTables t = tc_track_tables(m->pk.blob.data(), m->pk.L);
    for (int env = 0; env < n; env++)
        for (int j = 0; j < k; j++) out[(size_t)env * k + j] = tc_spawn_draw(t, rng_state + (size_t)env * TC_RNG_N, spawn_points, n_spawn_points);
}
// Generator.integers(0, high_excl) on n streams (tc_pcg_bounded), k draws each
HT_API void ht_pcg_bounded(int n, uint64_t *rng_state, uint32_t high_excl, int k, uint32_t *out) {
    for (int env = 0; env < n; env++)
        for (int j = 0; j < k; j++) out[(size_t)env * k + j] = tc_pcg_bounded(rng_state + (size_t)env * TC_RNG_N, high_excl);
}

// n Philox4x32-10 blocks: counters ctr [n,4], keys key [n,2] -> out [n,4]
HT_API void ht_philox(int n, const uint32_t *ctr, const uint32_t *key, uint32_t *out) {
    for (int i = 0; i < n; i++)
        tc_philox4x32_10(ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3], key[2 * i], key[2 * i + 1], out + 4 * i);
}

// the fill phase of tc_noise_blobs_kernel with its 256 threads replayed as one: inside the disc hw of radius rad at (x, y),
// clipped to [H,W], dst |= sp (copy) or dst = 0
static void ht_blob_fill(uint8_t *dst, const uint8_t *sp, int H, int W, int x, int y, int rad, bool copy, const int *hw) {
    const int side = 2 * rad + 1;
    for (int i = 0; i < side * side; i++) {
        int ry = i / side - rad, rx = i % side - rad;
        int h = hw[ry < 0 ? -ry : ry];
        if (h < 0 || rx < -h || rx > h) continue;
        int px = x + rx, py = y + ry;
        if ((unsigned)px >= (unsigned)W || (unsigned)py >= (unsigned)H) continue;
        size_t o = (size_t)py * W + px;
        if (copy) dst[o] |= sp[o];
        else dst[o] = 0;
    }
}

// cv2.circle(img, (x, y), radius, 255, -1) on a zero img [H,W] through tc_circle_halfwidths and the kernel's fill (radius < 1024)
HT_API void ht_circle(uint8_t *img, int H, int W, int x, int y, int radius) {
    int hw[1024];
    tc_circle_halfwidths(radius, hw);
    std::vector<uint8_t> ones((size_t)H * W, 255);
    ht_blob_fill(img, ones.data(), H, W, x, y, radius, true, hw);
}

// mirrors tc_noise_blobs_kernel over obs [n*n_cams, C, H, W] u8 in place (mask: optional, per env)
HT_API void ht_noise_blobs(uint8_t *obs, int n, int n_cams, int C, int H, int W, uint64_t seed, uint32_t step, int n_blobs, int max_radius,
                           int32_t env_index_offset, const uint8_t *mask) {
    int hw[1024];
    const size_t plane = (size_t)H * W;
    for (int v = 0; v < n * n_cams; v++) {
        const int env = v / n_cams, cam = v % n_cams;
        if (mask && !mask[env]) continue;
        uint8_t *base = obs + (size_t)v * C * plane;
        for (int c = 0; c < C; c++)
            for (int k = 0; k < n_blobs; k++) {
                const TcBlobDraw d = tc_noise_draw((uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)env + (uint32_t)env_index_offset, step, c, k, cam,
                                                   n_blobs, max_radius, H, W, C);
                tc_circle_halfwidths(d.radius, hw);
                if (!(d.copy && d.src == c)) ht_blob_fill(base + (size_t)c * plane, base + (size_t)d.src * plane, H, W, d.x, d.y, d.radius, d.copy != 0, hw);
            }
    }
}

// ---- visible-set tables (tc_cull.h): the camera pass of tc_render_env_kernel on the sub-graph of the camera's ground cell
struct HtCull { TcCull c; };
HT_API HtCull *ht_cull_create(const TcMapDesc *map, double radius, double cell, double margin) {
    HtCull *h = new HtCull();
    tc_build_cull(map, radius, cell, margin, h->c);
    return h;
}
HT_API void ht_cull_destroy(HtCull *h) { delete h; }
HT_API void ht_cull_info(const HtCull *h, double *out6) {
    out6[0] = h->c.radius; out6[1] = (double)h->c.desc.size(); out6[2] = h->c.mean_nodes; out6[3] = h->c.max_nodes;
    out6[4] = h->c.grid.nx; out6[5] = h->c.grid.ny;
}
HT_API double ht_cull_radius_of(const double *cam_row, int H, int W) { return tc_cull_radius_of(cam_row, H, W); }

// mirrors the geometry phase of tc_render_env_kernel; output in the layout of ht_render's segment arrays (per class, list order)
HT_API void ht_project_culled(const HtMap *m, const HtCull *hc, int n, int H, int W, const double *pose, const double *cam, int32_t *seg_count,
                              int32_t *seg, int32_t *cell_nodes /* optional [n] */) {
    const int C = m->C;
    for (int env = 0; env < n; env++) {
        const double *ps = pose + (size_t)env * 12, *cm = cam + (size_t)env * TC_CAM_N;
        const TcCellBlob d = hc->c.desc[tc_cull_cell(hc->c.grid, ps)];
        if (cell_nodes) cell_nodes[env] = d.n_nodes;
        for (int c = 0; c < C; c++) seg_count[(size_t)env * C + c] = 0;
        if (d.n_nodes == 0) continue;
        const unsigned char *base = hc->c.blob.data() + d.offset;
        const TcClassTables ct = tc_class_tables_from_cell(base, d);
        const uint8_t *core = base + d.off_core, *edge_cls = base + d.off_edge_cls;
        const int nn = d.n_nodes, mm = d.n_edges;
        std::vector<double> Px(nn + 1), Py(nn + 1), Pz(nn + 1);
        std::vector<int32_t> ix(nn + 1), iy(nn + 1);
        std::vector<uint8_t> fA(nn + 1), fB(nn + 1), rA(nn + 1), rB(nn + 1), vis(nn + 1);
        TcProjScratch sc = {Px.data(), Py.data(), Pz.data(), ix.data(), iy.data(), fA.data(), rA.data(), vis.data()};
        const double max_range = cm[TC_CAM_MAX_RANGE];
        for (int v = 0; v < nn; v++) {
            tc_transform_node(ps, ct.nodes[2 * v], ct.nodes[2 * v + 1], Px[v], Py[v], Pz[v]);
            fA[v] = Pz[v] < 0;
        }
        for (int v = 0; v < nn; v++) fB[v] = fA[v] | (uint8_t)tc_clip_pass_node(ct, sc, fA.data(), v, true, -0.0000001);
        for (int v = 0; v < nn; v++) fA[v] = fB[v] | (uint8_t)tc_clip_pass_node(ct, sc, fB.data(), v, false, -0.0000001);
        for (int v = 0; v < nn; v++) rA[v] = Pz[v] > -max_range;
        for (int v = 0; v < nn; v++) rB[v] = rA[v] | (uint8_t)tc_clip_pass_node(ct, sc, rA.data(), v, true, -max_range);
        for (int v = 0; v < nn; v++) rA[v] = rB[v] | (uint8_t)tc_clip_pass_node(ct, sc, rB.data(), v, false, -max_range);
        for (int v = 0; v < nn; v++) {
            double u, w;
            tc_project(cm, Px[v], Py[v], Pz[v], u, w);
            ix[v] = tc_np_int32(u);
            iy[v] = tc_np_int32(w);
            vis[v] = (core[v] && u > 0 && u < W && w > 0 && w < H && fA[v] && rA[v]) ? 1 : 0;
        }
        for (int e = 0; e < mm; e++) {
            int n0 = ct.edges[2 * e], n1 = ct.edges[2 * e + 1];
            if (!(vis[n0] || vis[n1])) continue;
            const int c = edge_cls[e];
            int32_t *s = seg + ((size_t)env * m->sumE + m->edge_off[c] + seg_count[(size_t)env * C + c]++) * 4;
            s[0] = ix[n0]; s[1] = iy[n0]; s[2] = ix[n1]; s[3] = iy[n1];
        }
    }
}

// nearest laneline edge per class for n positions: through the index (use_index != 0, lanes replayed one by one like a
// group of `nlanes`) or by the plain scan of all edges; cand_len (optional [n]) = candidates looked at in class 0
HT_API void ht_nearest(const HtMap *m, int n, const double *xy, int use_index, int nlanes, int32_t *out, int32_t *cand_len, double *info3) {
    TcTrackTables t = tc_track_tables(m->pk.blob.data(), m->pk.L);
    ht_attach_near(m, t, use_index != 0);
    if (info3) { info3[0] = (double)m->near.nx * m->near.ny; info3[1] = m->near.mean_len; info3[2] = m->near.max_len; }
    const int C = m->C;
    for (int i = 0; i < n; i++) {
        const double px = xy[2 * i], py = xy[2 * i + 1];
        const int cell = tc_near_cell(t, px, py);
        if (cand_len) cand_len[i] = cell >= 0 ? t.near_off[cell + 1] - t.near_off[cell] : -1;
        for (int c = 0; c < C; c++) {
            const double *nodes = t.ll_nodes + 2 * t.ll_node_off[c];
            const int32_t *edges = t.ll_edges + 2 * t.ll_edge_off[c];
            const int mm = t.ll_edge_off[c + 1] - t.ll_edge_off[c];
            int best = -1;
            double bd = 0;
            for (int lane = 0; lane < (nlanes > 0 ? nlanes : 1); lane++) {   // the group reduction: lexicographic (distance, edge)
                TcLanes g = {lane, nlanes > 0 ? nlanes : 1};
                int e;
                // a one-lane group per replayed lane: the lane's own candidates, no shuffle
                if (cell >= 0) {
                    const int32_t *o = t.near_off + (size_t)c * t.near_nx * t.near_ny + cell;
                    e = -1;
                    double d_e = 0;
                    for (int k = g.lane; k < o[1] - o[0]; k += g.n) {
                        int ee = t.near_edge[o[0] + k];
                        double d = fabs(tc_dist(px, py, nodes[2 * edges[2 * ee]], nodes[2 * edges[2 * ee] + 1]) +
                                        tc_dist(px, py, nodes[2 * edges[2 * ee + 1]], nodes[2 * edges[2 * ee + 1] + 1]));
                        if (e < 0 || d < d_e) { e = ee; d_e = d; }
                    }
                    if (e >= 0 && (best < 0 || d_e < bd || (d_e == bd && e < best))) { best = e; bd = d_e; }
                } else {
                    TcLanes g1 = {0, 1};
                    best = tc_nearest_edge(g1, nodes, edges, mm, px, py, nullptr, 0, 0);
                    break;
                }
            }
            out[(size_t)i * C + c] = best;
        }
    }
}
