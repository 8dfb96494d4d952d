// tc_core.cuh — the arithmetic of the hot path as lane-parallel __host__ __device__ code.
//
// Everything here is written once and compiled twice: by nvcc into the sm_100a kernels of libtinycarlo_b200.so
// (tc_kernels.cu: a warp per env for tracking, a block per (env, class) for the camera pass, a block per plane for
// rasterise+store), and by g++ into the CPU-only test library libtc_hosttest.so (tc_hosttest.cpp), where a "group"
// is one lane, so the parallel formulations can be checked in a container without a GPU. The product never loads
// the host build.
//
// Floating point: the reference computes in float64 with numpy/BLAS; parity needs the same operation order.
// Built with -fmad=false (nvcc) / -ffp-contract=off (g++): a*b+c is never fused implicitly, and the places where the
// reference's OpenBLAS dgemm fuses (k-ordered FMA chains, probed on numpy 2.3.5) use fma() explicitly.
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/tinycarlo_b200.h"

#if defined(__CUDACC__)
#define TC_HD __host__ __device__ __forceinline__
#else
#define TC_HD inline
#endif

#define TC_PI 3.14159265358979323846
#define TC_MAX_CLASSES 16

// ------------------------------------------------------------------------------------------------ lane groups
// A group of cooperating lanes: a warp on the device, a single lane on the host.
struct TcLanes {
    int lane, n;
};

// lexicographic (value, index) minimum over the group; every lane receives the result. Ties -> lowest index
// (layer.py:44 `d.index(min(d))`). A NaN value ties with another NaN: a car whose position is NaN (a NaN action) has NaN
// distances to every edge, and the sequential scan keeps its first candidate. Without the tie each lane would keep its own
// first candidate, and the result would depend on the lane that stores it (lane 0 of a group, or the lane that asked a
// whole warp to scan for it in the thread-per-env kernel).
TC_HD void tc_group_argmin(const TcLanes &g, double &d, int &idx) {
#if defined(__CUDA_ARCH__)
    // groups are aligned power-of-two slices of a warp (32: warp-per-env tracking; 8: four envs per warp; 1: thread-per-env, where
    // the lane's own result is the group's): the xor butterfly below stays inside the slice
    unsigned lane_in_warp;
    asm("mov.u32 %0, %%laneid;" : "=r"(lane_in_warp));
    // only the group's own lanes take part: the groups of a warp follow different control flow (one env scans, its neighbour does not)
    const unsigned mask = g.n >= 32 ? 0xffffffffu : (((1u << g.n) - 1u) << (lane_in_warp & ~(unsigned)(g.n - 1)));
    for (int off = g.n >> 1; off > 0; off >>= 1) {
        double od = __shfl_xor_sync(mask, d, off);
        int oi = __shfl_xor_sync(mask, idx, off);
        if (oi >= 0 && (idx < 0 || od < d || ((od == d || (od != od && d != d)) && oi < idx))) {
            d = od;
            idx = oi;
        }
    }
#else
    (void)g; (void)d; (void)idx;
#endif
}

// ------------------------------------------------------------------------------------------------ small math
// helper.py:11-19
// (the reference's loops never end for +-inf and take |a|/2pi rounds: angles on this path are sums of a few values in
// [-pi, pi] and maneuver * pi/2, so anything beyond 1e4 rad is a non-finite or corrupt input and comes back as NaN,
// which every comparison downstream treats as "no")
TC_HD double tc_clip_angle(double a) {
    if (!(fabs(a) <= 1.0e4)) return NAN;
    while (a > TC_PI) a -= 2 * TC_PI;
    while (a < -TC_PI) a += 2 * TC_PI;
    return a;
}
// layer.py:187 (the reference squares with pow(x, 2.0); x*x is its correctly rounded value)
TC_HD double tc_dist(double ax, double ay, double bx, double by) {
    double dx = ax - bx, dy = ay - by;
    return sqrt(dx * dx + dy * dy);
}
// np.clip on float64 scalars (NaN propagates, as in numpy)
TC_HD double tc_np_clip(double x, double lo, double hi) {
    if (x != x) return x;
    double m = x > lo ? x : lo;
    return m < hi ? m : hi;
}
// numpy float64 -> int32 cast (renderer.py:43,50): truncation, NaN/inf/out of range -> INT_MIN (x86 cvttsd2si)
TC_HD int32_t tc_np_int32(double v) {
    if (!(v > -2147483649.0 && v < 2147483648.0)) return INT32_MIN;
    return (int32_t)v;
}

// ------------------------------------------------------------------------------------------------ map tables
// Views into the packed table blob (global memory, or the shared-memory copy a block staged with TMA).
struct TcTrackTables {
    int n_classes;
    int lp_n_nodes, lp_n_edges;
    const double *lp_nodes;      // [P][2]
    const double *lp_orient;     // [Q]
    const double *lp_orient_rev; // [Q]
    const double *ll_nodes;      // [sumN][2]
    const int32_t *lp_edges;     // [Q][2]
    const int32_t *next_off;     // [P+1] CSR over lanepath edges by start node (edge-list order, layer.py:183)
    const int32_t *next_edge;    // [Q]
    const int32_t *prev_off;     // [P+1] CSR by end node (layer.py:185)
    const int32_t *prev_edge;    // [Q]
    const int32_t *ll_edges;     // [sumE][2] class-local node ids
    const int32_t *ll_node_off;  // [C+1]
    const int32_t *ll_edge_off;  // [C+1]
    const float *ll_nodes32;     // [sumN][2] float copy of ll_nodes for the pre-filter of the nearest-edge scan
    double scan_margin;          // 2*eps of the float pre-filter (metres)
    double scan_limit;           // |x|, |y| up to which that margin is proven; farther out the scan is plain float64
    // nearest-laneline index (tc_cull.h tc_build_near; global memory, optional): per (class, ground cell) the edges that can
    // be the arg-min of d(p,n0)+d(p,n1) for a p inside the cell, ascending
    double near_x0, near_y0, near_inv_cell;
    int near_nx, near_ny;        // near_nx == 0: no index, scan all edges
    const int32_t *near_off;     // [C * nx * ny + 1]
    const uint16_t *near_edge;
};

// Byte offsets of the sections inside the blob (all multiples of 16); filled by the host at staging.
struct TcBlobLayout {
    int32_t n_classes, lp_n_nodes, lp_n_edges, sum_nodes, sum_edges;
    int32_t off_lp_nodes, off_lp_orient, off_lp_orient_rev, off_ll_nodes, off_lp_edges, off_next_off, off_next_edge, off_prev_off,
        off_prev_edge, off_ll_edges, off_ll_node_off, off_ll_edge_off, off_ll_nodes32;
    int32_t total_bytes;
    double scan_margin, scan_limit;
};

TC_HD TcTrackTables tc_track_tables(const unsigned char *base, const TcBlobLayout &L) {
    TcTrackTables t;
    t.n_classes = L.n_classes;
    t.lp_n_nodes = L.lp_n_nodes;
    t.lp_n_edges = L.lp_n_edges;
    t.lp_nodes = (const double *)(base + L.off_lp_nodes);
    t.lp_orient = (const double *)(base + L.off_lp_orient);
    t.lp_orient_rev = (const double *)(base + L.off_lp_orient_rev);
    t.ll_nodes = (const double *)(base + L.off_ll_nodes);
    t.lp_edges = (const int32_t *)(base + L.off_lp_edges);
    t.next_off = (const int32_t *)(base + L.off_next_off);
    t.next_edge = (const int32_t *)(base + L.off_next_edge);
    t.prev_off = (const int32_t *)(base + L.off_prev_off);
    t.prev_edge = (const int32_t *)(base + L.off_prev_edge);
    t.ll_edges = (const int32_t *)(base + L.off_ll_edges);
    t.ll_node_off = (const int32_t *)(base + L.off_ll_node_off);
    t.ll_edge_off = (const int32_t *)(base + L.off_ll_edge_off);
    t.ll_nodes32 = (const float *)(base + L.off_ll_nodes32);
    t.scan_margin = L.scan_margin;
    t.scan_limit = L.scan_limit;
    t.near_x0 = t.near_y0 = t.near_inv_cell = 0.0;
    t.near_nx = t.near_ny = 0;
    t.near_off = nullptr; t.near_edge = nullptr;
    return t;
}

// ------------------------------------------------------------------------------------------------ layer.py queries
// layer.py:105-124 over a CSR slice [b, e) of lanepath edges incident to `node` (forward: edges leaving it, else
// edges entering it). Returns the CSR position of the picked edge, -1 for None. The reference drops self-loops from
// the orientation list but indexes the unfiltered list with the winner; kept.
TC_HD int tc_pick_edge(const TcTrackTables &t, int node, double orientation, const int32_t *csr, int b, int e, bool forward) {
    int n = e - b;
    if (n == 0) return -1;
    if (n <= 1) return b;
    int k = 0, best = -1;
    double bd = 0;
    for (int i = b; i < e; i++) {
        int ed = csr[i];
        int nn = forward ? t.lp_edges[2 * ed + 1] : t.lp_edges[2 * ed];
        if (nn == node) continue;
        double o = forward ? t.lp_orient[ed] : t.lp_orient_rev[ed];
        double d = fabs(tc_clip_angle(o - orientation));
        if (best < 0 || d < bd) {
            best = k;
            bd = d;
        }
        k++;
    }
    if (best < 0) return -1;
    return b + best;
}

// layer.py:126-142 on explicit node coordinates. The reference tests |angle(p-n0) - angle(e)| <= pi/2 and
// |angle(p-n1) - angle(-e)| <= pi/2 through four atan2 calls; the angle between two vectors is within pi/2 iff their dot
// product is >= 0, and the two formulations can only disagree when the angle is within a few ulp of pi/2. The atan2
// evaluation is therefore kept for the near-perpendicular band (|cos| < 1e-9, which contains the exactly perpendicular
// cases of the reference's unit tests) and skipped everywhere else.
TC_HD bool tc_angle_within_half_pi(double ux, double uy, double vx, double vy) {
    double dot = ux * vx + uy * vy;
    double scale = (fabs(ux) + fabs(uy)) * (fabs(vx) + fabs(vy));
    if (fabs(dot) > 1e-9 * scale) return dot > 0;
    return fabs(tc_clip_angle(atan2(uy, ux) - atan2(vy, vx))) <= TC_PI / 2;
}
TC_HD bool tc_within_edge_bounds(double px, double py, double n0x, double n0y, double n1x, double n1y) {
    if (px == n0x && py == n0y) return true;
    if (px == n1x && py == n1y) return true;
    double ex = n1x - n0x, ey = n1y - n0y;
    return tc_angle_within_half_pi(px - n0x, py - n0y, ex, ey) && tc_angle_within_half_pi(px - n1x, py - n1y, -ex, -ey);
}
// layer.py:144-164
TC_HD double tc_distance_to_edge(double px, double py, double n1x, double n1y, double n2x, double n2y) {
    double lx = n2x - n1x, ly = n2y - n1y;
    double vx = px - n1x, vy = py - n1y;
    if (lx == 0) return ly > 0 ? px - n1x : n1x - px;
    return (vx * ly - vy * lx) / sqrt(lx * lx + ly * ly);
}
// layer.py:33-44 / 59-74: argmin over edges [0, m) of |d(p,n0)+d(p,n1)|, optionally restricted to lanepath edges whose
// orientation is within `lim` rad of `orientation`. Group-parallel; every lane gets the winner (-1: none).
TC_HD int tc_nearest_edge(const TcLanes &g, const double *nodes, const int32_t *edges, int m, double px, double py,
                          const double *orient, double orientation, double lim) {
    int best = -1;
    double bd = 0;
    for (int e = g.lane; e < m; e += g.n) {
        if (orient && !(fabs(tc_clip_angle(orient[e] - orientation)) <= lim)) continue;
        int a = edges[2 * e], b = edges[2 * e + 1];
        double d = fabs(tc_dist(px, py, nodes[2 * a], nodes[2 * a + 1]) + tc_dist(px, py, nodes[2 * b], nodes[2 * b + 1]));
        if (best < 0 || d < bd) {
            best = e;
            bd = d;
        }
    }
    tc_group_argmin(g, bd, best);
    return best;
}

// The same arg-min for the per-class laneline scans (car.py:58, the bulk of the tracking kernel's arithmetic), with a
// float pre-filter: every edge gets a float estimate d32 of d0+d1 (|d32 - d| <= eps), the group takes the minimum, and
// only edges with d32 <= min32 + margin (margin >= 2*eps) are evaluated in float64. The true arg-min e* satisfies
// d32(e*) <= d(e*) + eps <= d(e) + eps <= d32(e) + 2*eps for every e, so it and all its float64 ties are candidates:
// the result is exactly that of the full float64 scan at a fraction of the float64 square roots.
TC_HD int tc_nearest_edge_prefiltered(const TcLanes &g, const double *nodes, const float *nodes32, const int32_t *edges, int m, double px,
                                      double py, double margin) {
    // single pass: min32 is the running minimum of the estimates seen by this lane; an edge is evaluated in float64
    // when its estimate is within the margin of it. The lane's true arg-min always passes (its estimate is within 2*eps
    // of every other estimate of the lane), so every lane ends with its exact arg-min and the group reduction is exact.
    const float fx = (float)px, fy = (float)py, fm = (float)margin;
    float min32 = 3.0e38f;
    int best = -1;
    double bd = 0;
    for (int e = g.lane; e < m; e += g.n) {
        int a = edges[2 * e], b = edges[2 * e + 1];
        float ax = nodes32[2 * a] - fx, ay = nodes32[2 * a + 1] - fy, bx = nodes32[2 * b] - fx, by = nodes32[2 * b + 1] - fy;
        float d32 = sqrtf(ax * ax + ay * ay) + sqrtf(bx * bx + by * by);
        if (d32 <= min32 + fm) {
            double d = fabs(tc_dist(px, py, nodes[2 * a], nodes[2 * a + 1]) + tc_dist(px, py, nodes[2 * b], nodes[2 * b + 1]));
            if (best < 0 || d < bd) {
                best = e;
                bd = d;
            }
        }
        min32 = d32 < min32 ? d32 : min32;
    }
    tc_group_argmin(g, bd, best);
    return best;
}

// The same arg-min over a candidate list (ascending edge ids) that is known to contain every edge attaining the minimum:
// the lists of the nearest-laneline index are a few edges long, each lane evaluates at most one or two in float64.
TC_HD int tc_nearest_edge_list(const TcLanes &g, const double *nodes, const int32_t *edges, const uint16_t *list, int count, double px, double py) {
    int best = -1;
    double bd = 0;
    for (int i = g.lane; i < count; i += g.n) {
        int e = list[i];
        int a = edges[2 * e], b = edges[2 * e + 1];
        double d = fabs(tc_dist(px, py, nodes[2 * a], nodes[2 * a + 1]) + tc_dist(px, py, nodes[2 * b], nodes[2 * b + 1]));
        if (best < 0 || d < bd) {
            best = e;
            bd = d;
        }
    }
    tc_group_argmin(g, bd, best);
    return best;
}
// cell of the nearest-laneline index that holds (x, y), or -1 (no index, outside the grid, NaN)
TC_HD int tc_near_cell(const TcTrackTables &t, double x, double y) {
    if (t.near_nx == 0) return -1;
    double fx = floor((x - t.near_x0) * t.near_inv_cell), fy = floor((y - t.near_y0) * t.near_inv_cell);
    if (!(fx >= 0 && fx < t.near_nx && fy >= 0 && fy < t.near_ny)) return -1;
    return (int)fy * t.near_nx + (int)fx;
}

// ------------------------------------------------------------------------------------------------ car.py
struct TcCarState {
    double x, y, rot, steer, vel, fx, fy;
    int path_len, last_man;
    int pn[8]; // local_path node pairs
    int pe[4]; // local_path edge ids
};

TC_HD void tc_load_state(const double *sf, const int32_t *si, TcCarState &s) {
    s.x = sf[TC_SF_X]; s.y = sf[TC_SF_Y]; s.rot = sf[TC_SF_ROT]; s.steer = sf[TC_SF_STEER_DEG]; s.vel = sf[TC_SF_VEL];
    s.fx = sf[TC_SF_FRONT_X]; s.fy = sf[TC_SF_FRONT_Y];
    s.path_len = si[TC_SI_PATH_LEN]; s.last_man = si[TC_SI_LAST_MANEUVER];
    for (int i = 0; i < 8; i++) s.pn[i] = si[TC_SI_PATH_NODES + i];
    for (int i = 0; i < 4; i++) s.pe[i] = si[TC_SI_PATH_EDGES + i];
}
TC_HD void tc_store_state(double *sf, int32_t *si, const TcCarState &s) {
    sf[TC_SF_X] = s.x; sf[TC_SF_Y] = s.y; sf[TC_SF_ROT] = s.rot; sf[TC_SF_STEER_DEG] = s.steer; sf[TC_SF_VEL] = s.vel;
    sf[TC_SF_FRONT_X] = s.fx; sf[TC_SF_FRONT_Y] = s.fy; sf[TC_SF_PAD] = 0.0;
    si[TC_SI_PATH_LEN] = s.path_len; si[TC_SI_LAST_MANEUVER] = s.last_man;
    for (int i = 0; i < 8; i++) si[TC_SI_PATH_NODES + i] = s.pn[i];
    for (int i = 0; i < 4; i++) si[TC_SI_PATH_EDGES + i] = s.pe[i];
    si[14] = 0; si[15] = 0;
}

// car.py:127-148 in three pieces, so that the one O(E) part - the u-turn's global scan - can be run by whichever lanes
// the caller has (the env's own group, or a whole warp on behalf of one of its envs when the kernel is thread-per-env):
//   tc_path_valid            the env tracks an edge (it was reset successfully)
//   tc_wants_uturn_scan      this step starts a u-turn (car.py:130)
//   tc_uturn_direction       the direction the scan filters by (car.py:128)
//   tc_find_local_path_given the rest, given the scan's result. Returns truncated.
TC_HD bool tc_path_valid(const TcTrackTables &t, const TcCarState &s) {
    // an env that was never reset (or whose reset found no successor edge) has no tracked edge: truncated, tables untouched
    return !(s.path_len <= 0 || s.pe[0] < 0 || s.pe[0] >= t.lp_n_edges || s.pn[0] < 0 || s.pn[1] < 0);
}
TC_HD bool tc_wants_uturn_scan(const TcTrackTables &t, const TcCarState &s, int maneuver) {
    return tc_path_valid(t, s) && maneuver == 2 && s.last_man != 2;
}
TC_HD double tc_uturn_direction(const TcTrackTables &t, const TcCarState &s, int maneuver) {
    return tc_clip_angle(t.lp_orient[s.pe[0]] + maneuver * TC_PI / 2);
}
TC_HD int tc_uturn_scan(const TcLanes &g, const TcTrackTables &t, double fx, double fy, double dir) {
    return tc_nearest_edge(g, t.lp_nodes, t.lp_edges, t.lp_n_edges, fx, fy, t.lp_orient, dir, 30.0 * (TC_PI / 180.0));
}
TC_HD bool tc_find_local_path_given(const TcTrackTables &t, TcCarState &s, int maneuver, int uturn_edge) {
    if (!tc_path_valid(t, s)) return true;
    double dir = tc_clip_angle(t.lp_orient[s.pe[0]] + maneuver * TC_PI / 2);
    int ne; // new first edge
    if (maneuver == 2 && s.last_man != 2) {
        ne = uturn_edge;
        dir = tc_clip_angle(dir + TC_PI);
        // reference: local_path=[None] -> TypeError at car.py:144. Here: truncated, path untouched (see DESIGN.md).
        if (ne < 0) return true;
    } else {
        // layer.py:77-103
        int e0 = s.pn[0], e1 = s.pn[1];
        int pn = tc_pick_edge(t, e1, dir, t.next_edge, t.next_off[e1], t.next_off[e1 + 1], true);
        int pp = tc_pick_edge(t, e0, dir, t.prev_edge, t.prev_off[e0], t.prev_off[e0 + 1], false);
        if (pn < 0 || pp < 0) return true;
        int en = t.next_edge[pn], ep = t.prev_edge[pp];
        int next_node = t.lp_edges[2 * en + 1], prev_node = t.lp_edges[2 * ep];
        double d0 = tc_dist(s.fx, s.fy, t.lp_nodes[2 * e0], t.lp_nodes[2 * e0 + 1]);
        double d1 = tc_dist(s.fx, s.fy, t.lp_nodes[2 * e1], t.lp_nodes[2 * e1 + 1]);
        double dn = tc_dist(s.fx, s.fy, t.lp_nodes[2 * next_node], t.lp_nodes[2 * next_node + 1]);
        double dp = tc_dist(s.fx, s.fy, t.lp_nodes[2 * prev_node], t.lp_nodes[2 * prev_node + 1]);
        if (dn < d0 && dn < d1) ne = en;
        else if (dp < d0 && dp < d1) ne = ep;
        else ne = s.pe[0];
    }
    s.last_man = maneuver;
    s.pe[0] = ne;
    s.pn[0] = t.lp_edges[2 * ne];
    s.pn[1] = t.lp_edges[2 * ne + 1];
    s.path_len = 1;
    for (int k = 0; k < 3; k++) {
        int from = s.vel > 0 ? s.pn[2 * (s.path_len - 1) + 1] : s.pn[2 * (s.path_len - 1)];
        int p = tc_pick_edge(t, from, dir, t.next_edge, t.next_off[from], t.next_off[from + 1], true);
        if (p < 0) return true;
        int e = t.next_edge[p];
        s.pe[s.path_len] = e;
        s.pn[2 * s.path_len] = from;
        s.pn[2 * s.path_len + 1] = t.lp_edges[2 * e + 1];
        s.path_len++;
    }
    return false;
}
// the env's own group does the scan (warp-per-env tracking, host test build)
TC_HD bool tc_find_local_path(const TcLanes &g, const TcTrackTables &t, TcCarState &s, int maneuver) {
    int ut = -1;
    if (tc_wants_uturn_scan(t, s, maneuver)) ut = tc_uturn_scan(g, t, s.fx, s.fy, tc_uturn_direction(t, s, maneuver));
    return tc_find_local_path_given(t, s, maneuver, ut);
}

// car.py:70-125 without the path update (v_cmd, s_cmd already clipped to [-1,1], env.py:118). cp = car parameter row.
TC_HD void tc_car_move(const double *cp, TcCarState &s, double v_cmd, double s_cmd) {
    double dt = cp[TC_CP_DT];
    double nv = v_cmd * cp[TC_CP_MAX_VELOCITY];
    if (!isnan(cp[TC_CP_MAX_ACCELERATION]))
        nv = tc_np_clip(nv, s.vel - cp[TC_CP_MAX_DECELERATION] * dt, s.vel + cp[TC_CP_MAX_ACCELERATION] * dt);
    s.vel = nv;
    double ns = s_cmd * cp[TC_CP_MAX_STEERING_DEG];
    if (!isnan(cp[TC_CP_STEERING_SPEED])) ns = tc_np_clip(ns, s.steer - cp[TC_CP_STEERING_SPEED] * dt, s.steer + cp[TC_CP_STEERING_SPEED] * dt);
    s.steer = ns;
    double vxn = cos(s.rot), vyn = sin(s.rot);
    if (fabs(s.steer) < 0.0001) {
        s.x = s.x + s.vel * vxn * dt;
        s.y = s.y + s.vel * vyn * dt;
    } else {
        double radius = cp[TC_CP_WHEELBASE] / tan(s.steer * (TC_PI / 180.0));
        double ang_vel = s.vel / radius;
        double dyaw = ang_vel * dt;
        double tx = vyn * radius, ty = -vxn * radius;
        double c = cos(dyaw), sn = sin(dyaw);
        // R_M.dot([tx, ty]) is an OpenBLAS dgemv: out_i = fma(R_i0, tx, R_i1 * ty)
        double r0 = fma(c, tx, (-sn) * ty);
        double r1 = fma(sn, tx, c * ty);
        s.x = s.x - tx + r0;
        s.y = s.y - ty + r1;
        s.rot += dyaw;
        if (s.rot > TC_PI) s.rot -= 2 * TC_PI;
        else if (s.rot < -TC_PI) s.rot += 2 * TC_PI;
    }
    s.fx = s.x + cp[TC_CP_WHEELBASE] * cos(s.rot);
    s.fy = s.y + cp[TC_CP_WHEELBASE] * sin(s.rot);
}
// car.py:70-125. Returns truncated.
TC_HD bool tc_car_step(const TcLanes &g, const TcTrackTables &t, const double *cp, TcCarState &s, double v_cmd, double s_cmd,
                       int maneuver) {
    tc_car_move(cp, s, v_cmd, s_cmd);
    return tc_find_local_path(g, t, s, maneuver);
}

// car.py:34-44 + map.py:66-68 with the spawn node drawn by the caller; spawn_rot/spawn_edge are host tables
// (first outgoing edge and its atan2). Returns false when the node has no successor (state untouched).
TC_HD bool tc_car_reset(const TcTrackTables &t, const double *cp, TcCarState &s, int node) {
    if (node < 0 || node >= t.lp_n_nodes || t.next_off[node] == t.next_off[node + 1]) return false;
    int e = t.next_edge[t.next_off[node]];
    s.x = t.lp_nodes[2 * node];
    s.y = t.lp_nodes[2 * node + 1];
    s.rot = t.lp_orient[e];
    s.steer = 0.0;
    s.vel = 0.0;
    s.fx = s.x + cp[TC_CP_WHEELBASE] * cos(s.rot);
    s.fy = s.y + cp[TC_CP_WHEELBASE] * sin(s.rot);
    s.path_len = 1;
    s.last_man = 0;
    for (int i = 0; i < 8; i++) s.pn[i] = -1;
    for (int i = 0; i < 4; i++) s.pe[i] = -1;
    s.pe[0] = e;
    s.pn[0] = node;
    s.pn[1] = t.lp_edges[2 * e + 1];
    return true;
}

// car.py:46-68 + env.py:83-99. Every lane returns the same values. dist/nearest have n_classes entries.
struct TcInfo {
    double cte, heading, velocity, reward;
    bool terminated;
};
// the nearest laneline edge of class c for a car at (x, y) whose ground cell has no candidate list: a scan over all edges
TC_HD int tc_nearest_laneline_scan(const TcLanes &g, const TcTrackTables &t, int c, double x, double y) {
    const double *nodes = t.ll_nodes + 2 * t.ll_node_off[c];
    const int32_t *edges = t.ll_edges + 2 * t.ll_edge_off[c];
    const int m = t.ll_edge_off[c + 1] - t.ll_edge_off[c];
    if (fabs(x) <= t.scan_limit && fabs(y) <= t.scan_limit)
        return tc_nearest_edge_prefiltered(g, nodes, t.ll_nodes32 + 2 * t.ll_node_off[c], edges, m, x, y, t.scan_margin);
    return tc_nearest_edge(g, nodes, edges, m, x, y, nullptr, 0, 0);   // a runaway car (wrapped envs never terminate): no pre-filter
}
// pre_nearest (optional): the nearest edge of every class, found by the caller (thread-per-env tracking: a warp scans on behalf
// of the env whose car left the index grid); otherwise the group looks it up / scans itself.
TC_HD TcInfo tc_get_info(const TcLanes &g, const TcTrackTables &t, const double *cp, const TcCarState &s, bool wrapped, double *dist,
                         int *nearest, const int *pre_nearest = nullptr) {
    TcInfo r;
    r.cte = 0; r.heading = 0; r.velocity = 0.0;
    for (int c = 0; c < t.n_classes; c++) { dist[c] = 0; nearest[c] = -1; }
    if (s.path_len >= 2) {
        int a = s.pn[2], b = s.pn[3];
        r.cte = tc_distance_to_edge(s.fx, s.fy, t.lp_nodes[2 * a], t.lp_nodes[2 * a + 1], t.lp_nodes[2 * b], t.lp_nodes[2 * b + 1]);
        r.heading = tc_clip_angle(t.lp_orient[s.pe[1]] - s.rot);
        const int cell = tc_near_cell(t, s.x, s.y);
        for (int c = 0; c < t.n_classes; c++) {
            const double *nodes = t.ll_nodes + 2 * t.ll_node_off[c];
            const int32_t *edges = t.ll_edges + 2 * t.ll_edge_off[c];
            int e;
            if (pre_nearest) e = pre_nearest[c];
            else if (cell >= 0) {
                const int32_t *o = t.near_off + (size_t)c * t.near_nx * t.near_ny + cell;
                e = tc_nearest_edge_list(g, nodes, edges, t.near_edge + o[0], o[1] - o[0], s.x, s.y);
            } else e = tc_nearest_laneline_scan(g, t, c, s.x, s.y);
            nearest[c] = e;
            if (e < 0) continue; // class without edges: the reference would raise on min([])
            int n0 = edges[2 * e], n1 = edges[2 * e + 1];
            double n0x = nodes[2 * n0], n0y = nodes[2 * n0 + 1], n1x = nodes[2 * n1], n1y = nodes[2 * n1 + 1];
            if (tc_within_edge_bounds(s.x, s.y, n0x, n0y, n1x, n1y)) dist[c] = fabs(tc_distance_to_edge(s.x, s.y, n0x, n0y, n1x, n1y));
            else {
                double da = tc_dist(s.x, s.y, n0x, n0y), db = tc_dist(s.fx, s.fy, n1x, n1y);
                dist[c] = db < da ? db : da;
            }
        }
        r.velocity = s.vel;
    }
    if (wrapped) { r.reward = 0; r.terminated = false; }
    else {
        double rw = (-1 / cp[TC_CP_TRACK_WIDTH]) * r.cte + 1;
        r.reward = 0 > rw ? 0 : rw;
        r.terminated = r.cte > (cp[TC_CP_TRACK_WIDTH] * 10);
    }
    return r;
}

// ------------------------------------------------------------------------------------------------ spawn draws
// map.py:51-69 on the device: numpy's Generator(PCG64(SeedSequence(seed))) stream of every env continues inside the reset
// path, so resets need no host round trip. State row (uint64 x 5): LCG state hi, lo, increment hi, lo, and the bit
// generator's buffered 32-bit half (bit 32 = valid, low 32 bits = value). Seeding (SeedSequence hashing, pcg64_srandom)
// stays on the host (tinycarlo_b200/pcg64.py); the stepping below is numpy's pcg64_next64 / pcg64_next32 /
// buffered_bounded_lemire_uint32, checked against numpy and against the reference's recorded draws.
TC_HD uint64_t tc_mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
TC_HD uint64_t tc_pcg_next64(uint64_t *st) {
    const uint64_t MH = 0x2360ED051FC65DA4ull, ML = 0x4385DF649FCCF645ull;
    uint64_t hi = st[TC_RNG_HI], lo = st[TC_RNG_LO];
    uint64_t plo = lo * ML;
    uint64_t phi = tc_mulhi64(lo, ML) + lo * MH + hi * ML;
    uint64_t nlo = plo + st[TC_RNG_INC_LO];
    uint64_t nhi = phi + st[TC_RNG_INC_HI] + (nlo < plo ? 1u : 0u);
    st[TC_RNG_HI] = nhi; st[TC_RNG_LO] = nlo;
    unsigned rot = (unsigned)(nhi >> 58);
    uint64_t x = nhi ^ nlo;
    return (x >> rot) | (x << ((64 - rot) & 63));
}
TC_HD uint32_t tc_pcg_next32(uint64_t *st) {
    if (st[TC_RNG_BUF] >> 32) {
        uint32_t v = (uint32_t)st[TC_RNG_BUF];
        st[TC_RNG_BUF] = 0;
        return v;
    }
    uint64_t v = tc_pcg_next64(st);
    st[TC_RNG_BUF] = (1ull << 32) | (v >> 32);
    return (uint32_t)v;
}
// Generator.integers(0, n) / the index of Generator.choice(seq of length n), n < 2^32
TC_HD uint32_t tc_pcg_bounded(uint64_t *st, uint32_t n) {
    if (n <= 1) return 0;
    const uint32_t rng = n - 1;
    if (rng == 0xFFFFFFFFu) return tc_pcg_next32(st);
    const uint64_t rng_excl = (uint64_t)rng + 1;
    uint64_t m = (uint64_t)tc_pcg_next32(st) * rng_excl;
    uint32_t leftover = (uint32_t)m;
    if (leftover < rng_excl) {
        const uint32_t threshold = (uint32_t)((0xFFFFFFFFu - rng) % rng_excl);
        while (leftover < threshold) {
            m = (uint64_t)tc_pcg_next32(st) * rng_excl;
            leftover = (uint32_t)m;
        }
    }
    return (uint32_t)(m >> 32);
}
// one spawn node: choice(spawn_points) or integers(0, n_nodes-1), redrawn while the node has no successor (map.py:61-64)
TC_HD int tc_spawn_draw(const TcTrackTables &t, uint64_t *st, const int32_t *choices, int n_choices) {
    for (int guard = 0; guard < 100000; guard++) {
        int node = n_choices > 0 ? choices[tc_pcg_bounded(st, (uint32_t)n_choices)] : (int)tc_pcg_bounded(st, (uint32_t)(t.lp_n_nodes - 1));
        if (node >= 0 && node < t.lp_n_nodes && t.next_off[node] != t.next_off[node + 1]) return node;
    }
    return -1;
}

// ------------------------------------------------------------------------------------------------ navigation goals
// tc_set_route's contract (include/tinycarlo_b200.h TcRouteDesc), one env at a time: tc_route_kernel runs it with a thread per
// env, ht_route_update sequentially. The route table comes from tc_route.h.
struct TcRoute {
    const double *D;        // [G][Q]
    const int8_t *cmd;      // [G][Q]
    const int32_t *goals;   // [G]
    int G, Q;
    double reach;
    int on_reach;
};
// the env's tracked edge pe0, or -1
TC_HD int tc_route_edge(const TcTrackTables &t, const int32_t *si) {
    const int pe = si[TC_SI_PATH_EDGES], pn0 = si[TC_SI_PATH_NODES], pn1 = si[TC_SI_PATH_NODES + 1];
    if (si[TC_SI_PATH_LEN] <= 0 || pe < 0 || pe >= t.lp_n_edges || pn0 < 0 || pn1 < 0 || pn1 >= t.lp_n_nodes) return -1;
    return pe;
}
// distance to goal k (+inf: no route, no tracked edge, no goal), with its command and reached flag
TC_HD double tc_route_eval(const TcTrackTables &t, const TcRoute &r, int pe, int pn1, double fx, double fy, int k, int &command,
                           bool &reached) {
    command = -1;
    reached = false;
    if (k < 0 || pe < 0) return INFINITY;
    const size_t at = (size_t)k * r.Q + pe;
    const double D = r.D[at];
    if (!(D < INFINITY)) return INFINITY;
    command = r.cmd[at];
    const double d = tc_dist(fx, fy, t.lp_nodes[2 * pn1], t.lp_nodes[2 * pn1 + 1]);
    reached = pn1 == r.goals[k] && d <= r.reach;
    return d + D;
}
// one draw among the valid goals (list order: finite D_k(pe0), not reached at this pose) on the goal stream; -1 when there is
// none, and then the stream does not move
TC_HD int tc_route_draw(const TcTrackTables &t, const TcRoute &r, int pe, int pn1, double fx, double fy, uint64_t *st) {
    if (pe < 0) return -1;
    const bool at_pn1 = tc_dist(fx, fy, t.lp_nodes[2 * pn1], t.lp_nodes[2 * pn1 + 1]) <= r.reach;
    uint32_t n = 0;
    for (int k = 0; k < r.G; k++) n += r.D[(size_t)k * r.Q + pe] < INFINITY && !(at_pn1 && r.goals[k] == pn1);
    if (n == 0) return -1;
    uint32_t j = tc_pcg_bounded(st, n);
    for (int k = 0; k < r.G; k++)
        if (r.D[(size_t)k * r.Q + pe] < INFINITY && !(at_pn1 && r.goals[k] == pn1)) {
            if (j == 0) return k;
            j--;
        }
    return -1;
}
// mode 0: after a step (draws where the step autoreset, resamples or terminates on a reach); 1: draw; 2: recompute with
// progress 0. k and prev are the env's goal index and prev_distance, updated in place; terminate: OR 1 into the done flags.
TC_HD void tc_route_update(const TcTrackTables &t, const TcRoute &r, int mode, bool was_reset, const int32_t *si, double fx, double fy,
                           uint64_t *st, int32_t &k, double &prev, int &command, double &distance, double &progress, bool &reached,
                           bool &terminate) {
    const int pe = tc_route_edge(t, si), pn1 = si[TC_SI_PATH_NODES + 1];
    if (k < 0 || k >= r.G) k = -1;
    progress = 0;
    reached = terminate = false;
    bool draw = mode == 1 || (mode == 0 && was_reset);
    if (!draw) {
        distance = tc_route_eval(t, r, pe, pn1, fx, fy, k, command, reached);
        if (mode == 0) {
            if (isfinite(prev) && isfinite(distance)) progress = prev - distance;
            if (reached) {
                if (r.on_reach == TC_ROUTE_TERMINATE) terminate = true;
                else draw = true;   // progress and reached stay those of the goal just reached
            }
        }
    }
    if (draw) {
        bool unused;
        k = tc_route_draw(t, r, pe, pn1, fx, fy, st);
        distance = tc_route_eval(t, r, pe, pn1, fx, fy, k, command, unused);   // a drawn goal is never reached where it was drawn
    }
    prev = distance;
}
TC_HD void tc_route_store(const TcTrackTables &t, const TcRoute &r, const TcRouteOutputs &o, size_t i, int k, int command, double distance,
                          double progress, bool reached) {
    const int node = k >= 0 ? r.goals[k] : -1;
    o.goal[i] = node;
    o.goal_position[2 * i] = node >= 0 ? (float)t.lp_nodes[2 * node] : NAN;
    o.goal_position[2 * i + 1] = node >= 0 ? (float)t.lp_nodes[2 * node + 1] : NAN;
    o.command[i] = command;
    o.distance[i] = (float)distance;
    o.progress[i] = (float)progress;
    o.reached[i] = reached ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------ blob noise
// NoiseObservationWrapper (tinycarlo/wrapper/observation.py:14-27) draws from the unseeded global numpy RNG; tc_noise_blobs
// draws every blob from Philox4x32-10 instead (contract in include/tinycarlo_b200.h), so the noise is a pure function of
// (seed, global env index, step, class, blob, camera), reproducible and independent of the sharding.
TC_HD void tc_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *out) {
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

struct TcBlobDraw {
    int x, y, radius, copy, src;
};
// blob `blob` of class c in camera `cam` of the env with global index env_global (counter word 2 wraps mod 2^32)
TC_HD TcBlobDraw tc_noise_draw(uint32_t seed_lo, uint32_t seed_hi, uint32_t env_global, uint32_t step, int c, int blob, int cam, int n_blobs,
                               int max_radius, int H, int W, int C) {
    uint32_t r[4];
    tc_philox4x32_10(env_global, step, (uint32_t)c * (uint32_t)n_blobs + (uint32_t)blob, (uint32_t)cam, seed_lo, seed_hi, r);
    TcBlobDraw d;
    d.x = (int)(r[0] % (uint32_t)W);
    d.y = (int)(r[1] % (uint32_t)H);
    d.radius = max_radius > 1 ? 1 + (int)(r[2] % (uint32_t)(max_radius - 1)) : 1;   // randint(1, max_radius)
    d.copy = (r[3] & 0xffffu) < 19661u;                                              // p = 0.3
    d.src = (int)((r[3] >> 16) % (uint32_t)C);
    return d;
}

// cv2.circle(img, centre, radius, colour, -1) is the filled midpoint circle: hw[|dy|] (dy = -radius..radius) = the half
// width of the disc's row dy, -1 for a row it does not reach. hw holds radius + 1 entries.
TC_HD void tc_circle_halfwidths(int radius, int *hw) {
    for (int i = 0; i <= radius; i++) hw[i] = -1;
    int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
    while (dx >= dy) {
        hw[dy] = hw[dy] > dx ? hw[dy] : dx;
        hw[dx] = hw[dx] > dy ? hw[dx] : dy;
        dy++; err += plus; plus += 2;
        int m = (err <= 0) - 1;
        err -= minus & m; dx += m; minus -= m & 2;
    }
}

// ------------------------------------------------------------------------------------------------ camera.py
// numpy matmul == OpenBLAS dgemm on these shapes: c_ij = fma(a_i3,b_3j, fma(a_i2,b_2j, fma(a_i1,b_1j, a_i0*b_0j)))
TC_HD void tc_mm_chain(const double *A, int ar, int ac, const double *B, int bc, double *C) {
    for (int i = 0; i < ar; i++)
        for (int j = 0; j < bc; j++) {
            double s = A[i * ac] * B[j];
            for (int k = 1; k < ac; k++) s = fma(A[i * ac + k], B[k * bc + j], s);
            C[i * bc + j] = s;
        }
}
// camera.py:61 with car.py:159-165: pose = E @ (Rz(-rot) @ T(-pos)); cr/sr = cos(rot)/sin(rot) (cos(-r)=cos r, sin(-r)=-sin r)
TC_HD void tc_camera_pose(const double *E, double x, double y, double cr, double sr, double *pose) {
    double c = cr, s = -sr;
    double R[16] = {c, -s, 0, 0, s, c, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    double T[16] = {1, 0, 0, -x, 0, 1, 0, -y, 0, 0, 1, 0, 0, 0, 0, 1};
    double M[16];
    tc_mm_chain(R, 4, 4, T, 4, M);
    tc_mm_chain(E, 3, 4, M, 4, pose);
}
// camera.py:59,124-131: one node (x, y, 0, 1) through the 3x4 pose (dgemm FMA chain over k)
TC_HD void tc_transform_node(const double *pose, double x, double y, double &X, double &Y, double &Z) {
    double r[3];
    for (int i = 0; i < 3; i++) {
        double s = pose[4 * i] * x;
        s = fma(pose[4 * i + 1], y, s);
        s = fma(pose[4 * i + 2], 0.0, s);
        s = fma(pose[4 * i + 3], 1.0, s);
        r[i] = s;
    }
    X = r[0]; Y = r[1]; Z = r[2];
}
// camera.py:112-122: move `mv` along the edge towards `keep` onto the plane z = tz (NaN row when parallel)
TC_HD void tc_move_to_z(double kx, double ky, double kz, double &mx, double &my, double &mz, double tz) {
    double dx = kx - mx, dy = ky - my, dz = kz - mz;
    if (dz == 0) {
        mx = my = mz = NAN;
        return;
    }
    double tt = (tz - mz) / dz;
    double nx = mx + tt * dx, ny = my + tt * dy, nz = mz + tt * dz;
    mx = nx; my = ny; mz = nz;
}
// camera.py:89,133-142: K @ P (dgemm FMA chain, K = [[fx,0,cx],[0,fy,cy],[0,0,1]]) / row 2
TC_HD void tc_project(const double *cam, double X, double Y, double Z, double &u, double &v) {
    double h0 = fma(cam[TC_CAM_CX], Z, fma(0.0, Y, cam[TC_CAM_FX] * X));
    double h1 = fma(cam[TC_CAM_CY], Z, fma(cam[TC_CAM_FY], Y, 0.0 * X));
    double h2 = fma(1.0, Z, fma(0.0, Y, 0.0 * X));
    u = h0 / h2;
    v = h1 / h2;
}

// Per-class tables for the camera pass (global memory).
struct TcClassTables {
    int n_nodes, n_edges;
    const double *nodes;    // [n][2]
    const int32_t *edges;   // [m][2]
    const int32_t *out_off; // [n+1] CSR: edges leaving a node, in edge order
    const int32_t *out_edge;
    const int32_t *in_off; // [n+1] CSR: edges entering a node, in edge order
    const int32_t *in_edge;
};

// A class's tables packed back to back for one TMA bulk copy into shared memory (sections 16-byte aligned):
// [nodes n*16][edges m*8][out_off (n+1)*4][out_edge m*4][in_off (n+1)*4][in_edge m*4]
struct TcClassBlob {
    int32_t n_nodes, n_edges;
    int32_t offset; // byte offset of this class inside the class-blob buffer
    int32_t bytes;  // multiple of 16
    int32_t off_edges, off_out_off, off_out_edge, off_in_off, off_in_edge; // relative to `offset`
};
TC_HD TcClassTables tc_class_tables_from_blob(const unsigned char *base, const TcClassBlob &b) {
    TcClassTables ct;
    ct.n_nodes = b.n_nodes; ct.n_edges = b.n_edges;
    ct.nodes = (const double *)base;
    ct.edges = (const int32_t *)(base + b.off_edges);
    ct.out_off = (const int32_t *)(base + b.off_out_off);
    ct.out_edge = (const int32_t *)(base + b.off_out_edge);
    ct.in_off = (const int32_t *)(base + b.off_in_off);
    ct.in_edge = (const int32_t *)(base + b.off_in_edge);
    return ct;
}

// Visible-set tables of the block-per-env render kernel (built by tc_cull.h, which also states why the result is unchanged):
// the sub-graph of the union of all classes that a camera standing in one ground cell can see. Same sections as a class
// blob plus a per-node "core" byte (only core nodes may be visible) and a per-edge class byte.
struct TcCellBlob {
    int32_t n_nodes, n_edges;
    int32_t offset, bytes; // inside the cell-blob buffer; bytes is a multiple of 16 (0: empty cell)
    int32_t off_edges, off_out_off, off_out_edge, off_in_off, off_in_edge, off_core, off_edge_cls;
};
struct TcCullGrid {
    double x0, y0, inv_cell;
    int32_t nx, ny; // nx == 0: culling off, descriptor 0 is the whole graph; descriptor nx*ny is the empty one (outside the grid)
};
// descriptor index for a camera whose world->camera pose is the row-major 3x4 [R|t]: the camera centre is -R^T t
TC_HD int tc_cull_cell(const TcCullGrid &g, const double *pose) {
    if (g.nx == 0) return 0;
    double cx = -(pose[0] * pose[3] + pose[4] * pose[7] + pose[8] * pose[11]);
    double cy = -(pose[1] * pose[3] + pose[5] * pose[7] + pose[9] * pose[11]);
    double fx = floor((cx - g.x0) * g.inv_cell), fy = floor((cy - g.y0) * g.inv_cell);
    if (!(fx >= 0 && fx < g.nx && fy >= 0 && fy < g.ny)) return g.nx * g.ny; // also NaN poses: nothing is visible
    return (int)fy * g.nx + (int)fx;
}
TC_HD TcClassTables tc_class_tables_from_cell(const unsigned char *base, const TcCellBlob &b) {
    TcClassTables ct;
    ct.n_nodes = b.n_nodes; ct.n_edges = b.n_edges;
    ct.nodes = (const double *)base;
    ct.edges = (const int32_t *)(base + b.off_edges);
    ct.out_off = (const int32_t *)(base + b.off_out_off);
    ct.out_edge = (const int32_t *)(base + b.off_out_edge);
    ct.in_off = (const int32_t *)(base + b.off_in_off);
    ct.in_edge = (const int32_t *)(base + b.off_in_edge);
    return ct;
}

// Scratch of one camera pass (shared memory on the device).
struct TcProjScratch {
    double *Px, *Py, *Pz; // [n]
    int32_t *ix, *iy;     // [n] projected coordinates after the int32 cast
    uint8_t *front, *inr, *vis; // [n]
};

// One of the four ordered clip passes of camera.py:70-86 in node-parallel form. In the reference each pass walks a
// list of edges fixed before the pass and moves one endpoint per edge, in edge order. All moves of a pass write nodes
// whose flag is clear and read nodes whose flag is set, so moves of different nodes commute; for one node the edges
// apply in CSR (= edge-list) order. `outgoing`: the moved node is e[0] (passes 1 and 3), else e[1] (passes 2 and 4).
// Caller synchronises the group before and after; flags are updated in tc_clip_pass_commit after the sync.
TC_HD bool tc_clip_pass_node(const TcClassTables &ct, const TcProjScratch &sc, const uint8_t *flag, int v, bool outgoing, double tz) {
    if (flag[v]) return false;
    const int32_t *off = outgoing ? ct.out_off : ct.in_off;
    const int32_t *lst = outgoing ? ct.out_edge : ct.in_edge;
    bool moved = false;
    double mx = sc.Px[v], my = sc.Py[v], mz = sc.Pz[v];
    for (int i = off[v]; i < off[v + 1]; i++) {
        int e = lst[i];
        int w = outgoing ? ct.edges[2 * e + 1] : ct.edges[2 * e];
        if (!flag[w]) continue;
        tc_move_to_z(sc.Px[w], sc.Py[w], sc.Pz[w], mx, my, mz, tz);
        moved = true;
    }
    if (moved) { sc.Px[v] = mx; sc.Py[v] = my; sc.Pz[v] = mz; }
    return moved;
}

// ------------------------------------------------------------------------------------------------ cv2.polylines
// Rasterisation into a flat 1-bit plane: bit index = y*W + x, 32-bit words. SURVEY.md Appendix A (OpenCV 4.13.0,
// LINE_8, shift 0, thickness t, 2-point open polyline with both caps). The scalar set-up (pre-clip, quad, walker
// events) is computed redundantly by every lane; pixels are spread over the lanes through closed forms of the
// incremental loops (all integer, hence exact).
#define TC_XY_SHIFT 16
#define TC_XY_ONE (1 << TC_XY_SHIFT)

struct TcPlane {
    uint32_t *bits; // flat bit plane
    int H, W;
    int y_lo, y_hi; // rows [y_lo, y_hi) of the frame may be drawn
    int row_base;   // bit index = (y - row_base)*W + x: y_lo for a band plane, -c*H for class c of a stacked C*H-row plane
};

TC_HD void tc_or_word(uint32_t *p, uint32_t m) {
#if defined(__CUDA_ARCH__)
    atomicOr(p, m);
#else
    *p |= m;
#endif
}
TC_HD void tc_put(const TcPlane &pl, int64_t x, int64_t y) {
    if (x < 0 || x >= pl.W || y < pl.y_lo || y >= pl.y_hi) return;
    int64_t b = (y - pl.row_base) * pl.W + x;
    tc_or_word(pl.bits + (b >> 5), 1u << (b & 31));
}
// inclusive span, x already clipped to [0, W-1]
TC_HD void tc_hline(const TcPlane &pl, int y, int x1, int x2) {
    if (y < pl.y_lo || y >= pl.y_hi || x2 < x1) return;
    int b1 = (y - pl.row_base) * pl.W + x1, b2 = (y - pl.row_base) * pl.W + x2;
    int w1 = b1 >> 5, w2 = b2 >> 5;
    uint32_t m1 = 0xffffffffu << (b1 & 31), m2 = 0xffffffffu >> (31 - (b2 & 31));
    if (w1 == w2) tc_or_word(pl.bits + w1, m1 & m2);
    else {
        tc_or_word(pl.bits + w1, m1);
        for (int w = w1 + 1; w < w2; w++) tc_or_word(pl.bits + w, 0xffffffffu);
        tc_or_word(pl.bits + w2, m2);
    }
}

TC_HD bool tc_clip_line(int64_t w, int64_t h, int64_t &x1, int64_t &y1, int64_t &x2, int64_t &y2) {
    if (w <= 0 || h <= 0) return false;
    int64_t right = w - 1, bottom = h - 1;
    int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
    int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
        int64_t a;
        if (c1 & 12) {
            a = c1 < 8 ? 0 : bottom;
            x1 += (int64_t)((double)(a - y1) * (double)(x2 - x1) / (double)(y2 - y1));
            y1 = a;
            c1 = (x1 < 0) + (x1 > right) * 2;
        }
        if (c2 & 12) {
            a = c2 < 8 ? 0 : bottom;
            x2 += (int64_t)((double)(a - y2) * (double)(x2 - x1) / (double)(y2 - y1));
            y2 = a;
            c2 = (x2 < 0) + (x2 > right) * 2;
        }
        if ((c1 & c2) == 0 && (c1 | c2) != 0) {
            if (c1) {
                a = c1 == 1 ? 0 : right;
                y1 += (int64_t)((double)(a - x1) * (double)(y2 - y1) / (double)(x2 - x1));
                x1 = a;
                c1 = 0;
            }
            if (c2) {
                a = c2 == 1 ? 0 : right;
                y2 += (int64_t)((double)(a - x2) * (double)(y2 - y1) / (double)(x2 - x1));
                x2 = a;
                c2 = 0;
            }
        }
    }
    return (c1 | c2) == 0;
}

// Truncating integer division for |num| < 2^53 and 0 < |den| < 2^53 through one fp64 division: the correctly rounded
// quotient is off by at most |q|*2^-53 < 1/|den| <= the distance of a non-integer num/den to the next integer, so the
// truncation equals C's num / den. (64-bit integer division is ~4x more instructions on the GPU.)
TC_HD int64_t tc_div_trunc(int64_t num, int64_t den) { return (int64_t)((double)num / (double)den); }

// ---- primitives ----
// A polyline is first turned into a short list of drawing primitives by scalar code (tc_polyline_setup: the pre-clip,
// the quad, the clipped outline edges, the scan-line walker events; int64/double, a few hundred instructions, one
// thread per segment), then the primitives are drawn by lane-parallel loops (tc_prim_draw) whose per-pixel arithmetic
// is 32-bit. Everything after the pre-clip lies within [-t, W+t] x [-t, H+t] px, i.e. below 2^27 in 16.16.
enum { TC_PRIM_NONE = 0, TC_PRIM_LINE2 = 1, TC_PRIM_SPAN = 2, TC_PRIM_CIRCLE = 3, TC_PRIM_BRES = 4 };
#define TC_MAX_PRIMS_PER_SEG 12 // 4 outline edges + <= 6 fill spans + 2 caps
struct TcPrim {
    int32_t kind;
    int32_t a[7];
};

// thickness <= 1: LineIterator (8-connected, left to right). Step i of the Bresenham walk sits at major offset i and
// minor offset c_i = floor((2*dy*i + dx - 1) / (2*dx)) — the closed form of `err` staying in [-2dy, 2dx-2dy).
TC_HD int tc_setup_bresenham(int W, int H, int64_t x1, int64_t y1, int64_t x2, int64_t y2, TcPrim *out) {
    if (x1 < 0 || x1 >= W || x2 < 0 || x2 >= W || y1 < 0 || y1 >= H || y2 < 0 || y2 >= H)
        if (!tc_clip_line(W, H, x1, y1, x2, y2)) return 0;
    int64_t dx = x2 - x1, dy = y2 - y1;
    int sy = 1;
    if (dx < 0) { dx = -dx; dy = -dy; x1 = x2; y1 = y2; }
    if (dy < 0) { dy = -dy; sy = -1; }
    int vert = dy > dx;
    if (vert) { int64_t t = dx; dx = dy; dy = t; }
    out->kind = TC_PRIM_BRES;
    out->a[0] = vert; out->a[1] = (int32_t)x1; out->a[2] = (int32_t)y1; out->a[3] = sy; out->a[4] = (int32_t)dx; out->a[5] = (int32_t)dy;
    out->a[6] = 0;
    return 1;
}

// 16.16 DDA of one quad outline edge
TC_HD int tc_setup_line2(int W, int H, int64_t x1, int64_t y1, int64_t x2, int64_t y2, TcPrim *out) {
    if (!tc_clip_line((int64_t)W << TC_XY_SHIFT, (int64_t)H << TC_XY_SHIFT, x1, y1, x2, y2)) return 0;
    int64_t dx = x2 - x1, dy = y2 - y1, ax = dx < 0 ? -dx : dx, ay = dy < 0 ? -dy : dy, step, n;
    int xmajor = ax > ay;
    if (xmajor) {
        if (dx < 0) { dy = -dy; int64_t t; t = x1; x1 = x2; x2 = t; t = y1; y1 = y2; y2 = t; }
        step = tc_div_trunc(dy * TC_XY_ONE, ax | 1);
        n = (x2 - x1) >> TC_XY_SHIFT;
    } else {
        if (dy < 0) { dx = -dx; int64_t t; t = x1; x1 = x2; x2 = t; t = y1; y1 = y2; y2 = t; }
        step = tc_div_trunc(dx * TC_XY_ONE, ay | 1);
        n = (y2 - y1) >> TC_XY_SHIFT;
    }
    x1 += TC_XY_ONE >> 1;
    y1 += TC_XY_ONE >> 1;
    out->kind = TC_PRIM_LINE2;
    out->a[0] = xmajor;
    out->a[1] = (int32_t)(xmajor ? (x1 >> TC_XY_SHIFT) : (y1 >> TC_XY_SHIFT)); // integer start on the major axis
    out->a[2] = (int32_t)(xmajor ? y1 : x1);                                    // 16.16 start on the minor axis
    out->a[3] = (int32_t)step;
    out->a[4] = (int32_t)n;
    out->a[5] = (int32_t)((x2 + (TC_XY_ONE >> 1)) >> TC_XY_SHIFT); // the extra end-point pixel
    out->a[6] = (int32_t)((y2 + (TC_XY_ONE >> 1)) >> TC_XY_SHIFT);
    return 1;
}

// FillConvexPoly (4 vertices, shift 16). The scan-line loop only changes walker state on rows where a walker reaches
// the end of its polygon edge; between such rows x advances linearly. The (<= 6) events are replayed here and every
// run of rows becomes one SPAN primitive; the outline edges become LINE2 primitives.
// Fixed slots of a segment's primitive list: 0-3 outline edges, 4-9 fill spans, 10-11 caps (or slot 0: Bresenham line).
enum { TC_SLOT_EDGE0 = 0, TC_SLOT_SPAN0 = 4, TC_SLOT_CAP0 = 10 };
enum { TC_ROLE_SPANS = 0, TC_ROLE_EDGE0 = 1 /* ..4 */, TC_ROLE_CAPS = 5, TC_N_ROLES = 6, TC_ROLE_ALL = -1 };

// 4-way select instead of a runtime-indexed local array (which would live in local memory: on the GPU every such access
// queues behind the observation stores in the load/store pipeline)
TC_HD int64_t tc_sel4(int i, int64_t a, int64_t b, int64_t c, int64_t d) { return i == 0 ? a : (i == 1 ? b : (i == 2 ? c : d)); }

template <bool COMPACT>
TC_HD void tc_setup_fill_convex_poly4(int W, int H, const int64_t (*v)[2], int role, TcPrim *out) {
    const int npts = 4;
    const int64_t delta = TC_XY_ONE >> 1;
    const int64_t vx0 = v[0][0], vx1 = v[1][0], vx2 = v[2][0], vx3 = v[3][0];
    const int64_t vy0 = v[0][1], vy1 = v[1][1], vy2 = v[2][1], vy3 = v[3][1];
    int imin = 0, edges = npts;
    int64_t xmin = vx0, xmax = vx0, ymin = vy0, ymax = vy0;
    if (vy1 < ymin) { ymin = vy1; imin = 1; }
    if (vy2 < ymin) { ymin = vy2; imin = 2; }
    if (vy3 < ymin) { ymin = vy3; imin = 3; }
    ymax = vy1 > ymax ? vy1 : ymax; ymax = vy2 > ymax ? vy2 : ymax; ymax = vy3 > ymax ? vy3 : ymax;
    xmax = vx1 > xmax ? vx1 : xmax; xmax = vx2 > xmax ? vx2 : xmax; xmax = vx3 > xmax ? vx3 : xmax;
    xmin = vx1 < xmin ? vx1 : xmin; xmin = vx2 < xmin ? vx2 : xmin; xmin = vx3 < xmin ? vx3 : xmin;
    // outline: edge i runs from vertex i-1 to vertex i (the closing edge first)
    if (COMPACT) {
        // one instance of the edge set-up for the four edge roles (block-per-env kernel: the roles run concurrently on
        // different warps and its code should stay small); role is never TC_ROLE_ALL here
        if (role >= TC_ROLE_EDGE0 && role < TC_ROLE_EDGE0 + 4) {
            const int i = role - TC_ROLE_EDGE0;
            tc_setup_line2(W, H, tc_sel4(i, vx3, vx0, vx1, vx2), tc_sel4(i, vy3, vy0, vy1, vy2), tc_sel4(i, vx0, vx1, vx2, vx3),
                           tc_sel4(i, vy0, vy1, vy2, vy3), out + TC_SLOT_EDGE0 + i);
            return;
        }
        if (role != TC_ROLE_SPANS) return;
    } else {
    if (role == TC_ROLE_ALL || role == TC_ROLE_EDGE0 + 0) tc_setup_line2(W, H, vx3, vy3, vx0, vy0, out + TC_SLOT_EDGE0 + 0);
    if (role == TC_ROLE_ALL || role == TC_ROLE_EDGE0 + 1) tc_setup_line2(W, H, vx0, vy0, vx1, vy1, out + TC_SLOT_EDGE0 + 1);
    if (role == TC_ROLE_ALL || role == TC_ROLE_EDGE0 + 2) tc_setup_line2(W, H, vx1, vy1, vx2, vy2, out + TC_SLOT_EDGE0 + 2);
    if (role == TC_ROLE_ALL || role == TC_ROLE_EDGE0 + 3) tc_setup_line2(W, H, vx2, vy2, vx3, vy3, out + TC_SLOT_EDGE0 + 3);
    }
    if (role != TC_ROLE_ALL && role != TC_ROLE_SPANS) return;
    int k = TC_SLOT_SPAN0;
    xmin = (xmin + delta) >> TC_XY_SHIFT; xmax = (xmax + delta) >> TC_XY_SHIFT;
    ymin = (ymin + delta) >> TC_XY_SHIFT; ymax = (ymax + delta) >> TC_XY_SHIFT;
    if ((int)xmax < 0 || (int)ymax < 0 || (int)xmin >= W || (int)ymin >= H) return;
    if (ymax > H - 1) ymax = H - 1;
    int y = (int)ymin;
    // the two scan-line walkers (kept in scalars: e?0 walks the vertices upwards, e?1 downwards)
    int idxA = imin, idxB = imin, yeA = y, yeB = y;
    int64_t xA = -TC_XY_ONE, xB = -TC_XY_ONE, dxA = 0, dxB = 0;
    // A walker picks a polygon edge up on the scan line of the edge's start vertex (y == its rounded y: the loop below only stops
    // on vertex rows), and only edges that lead to a LATER row, so the slope it computes there is a function of the edge alone:
    // trunc(((xe - xs) * 2 + dy) / (2 * dy)), dy = the edge's rounded height in its downward direction. The block-per-env kernels
    // (COMPACT) compute the four slopes up front - four independent divisions the hardware overlaps - instead of one after the
    // other inside the data-dependent walk; the values, and therefore the spans, are the same (tests/test_core_host.py fuzzes both
    // formulations against the oracle).
    int64_t sl0 = 0, sl1 = 0, sl2 = 0, sl3 = 0;
    if (COMPACT) {
        const int ry0 = (int)((vy0 + delta) >> TC_XY_SHIFT), ry1 = (int)((vy1 + delta) >> TC_XY_SHIFT), ry2 = (int)((vy2 + delta) >> TC_XY_SHIFT),
                  ry3 = (int)((vy3 + delta) >> TC_XY_SHIFT);
#define TC_SLOPE(XA, RA, XB, RB) ((RB) == (RA) ? (int64_t)0 : ((RB) > (RA) ? tc_div_trunc(((XB) - (XA)) * 2 + ((RB) - (RA)), 2 * ((RB) - (RA))) \
                                                                        : tc_div_trunc(((XA) - (XB)) * 2 + ((RA) - (RB)), 2 * ((RA) - (RB)))))
        sl0 = TC_SLOPE(vx0, ry0, vx1, ry1);   // polygon edge k joins vertices k and k+1
        sl1 = TC_SLOPE(vx1, ry1, vx2, ry2);
        sl2 = TC_SLOPE(vx2, ry2, vx3, ry3);
        sl3 = TC_SLOPE(vx3, ry3, vx0, ry0);
#undef TC_SLOPE
    }
    while (true) {
#define TC_WALK(IDX, YE, X, DX, DI)                                                        \
        if (y >= YE) {                                                                     \
            int idx0 = IDX;                                                                \
            int idx = idx0 + DI;                                                           \
            if (idx >= npts) idx -= npts;                                                  \
            for (; edges-- > 0;) {                                                         \
                int ty = (int)((tc_sel4(idx, vy0, vy1, vy2, vy3) + delta) >> TC_XY_SHIFT); \
                if (ty > y) {                                                              \
                    int64_t xs = tc_sel4(idx0, vx0, vx1, vx2, vx3), xe = tc_sel4(idx, vx0, vx1, vx2, vx3); \
                    YE = ty;                                                               \
                    /* the polygon edge between idx0 and idx: the one with the smaller index, or edge 3 for the pair (3, 0) */ \
                    DX = COMPACT ? tc_sel4(DI == 1 ? idx0 : idx, sl0, sl1, sl2, sl3)      \
                                 : tc_div_trunc((xe - xs) * 2 + (ty - y), 2 * (ty - y));  \
                    X = xs;                                                                \
                    IDX = idx;                                                             \
                    break;                                                                 \
                }                                                                          \
                idx0 = idx;                                                                \
                idx += DI;                                                                 \
                if (idx >= npts) idx -= npts;                                              \
            }                                                                              \
        }
        TC_WALK(idxA, yeA, xA, dxA, 1)
        TC_WALK(idxB, yeB, xB, dxB, (npts - 1))
#undef TC_WALK
        if (edges < 0) break;
        // rows y .. y_end-1 share the walker state: the next event is the smaller ye (both are > y here), capped by ymax
        int y_end = yeA < yeB ? yeA : yeB;
        if (y_end > (int)ymax + 1) y_end = (int)ymax + 1;
        if (y_end <= y) y_end = y + 1;
        int r0 = y < 0 ? 0 : y;
        if (r0 < y_end && k < TC_SLOT_CAP0) {
            TcPrim &q = out[k++];
            q.kind = TC_PRIM_SPAN;
            q.a[0] = y; q.a[1] = r0; q.a[2] = y_end;
            q.a[3] = (int32_t)xA; q.a[4] = (int32_t)dxA; q.a[5] = (int32_t)xB; q.a[6] = (int32_t)dxB;
        }
        xA += (int64_t)(y_end - y) * dxA;
        xB += (int64_t)(y_end - y) * dxB;
        y = y_end;
        if (y > (int)ymax) break;
    }
}

TC_HD int64_t tc_cv_round(double v) { return (int64_t)rint(v); } // round half to even

// cv2.polylines(img, np.int32([[p0, p1]]), False, 255, t) -> primitives in the 12 fixed slots of `out` (the caller has
// set every slot to TC_PRIM_NONE). `role` selects which slots this call fills, so that the independent parts of one
// segment can be set up by different threads (each repeats the cheap pre-clip and quad construction): TC_ROLE_SPANS,
// TC_ROLE_EDGE0+i, TC_ROLE_CAPS, or TC_ROLE_ALL.
template <bool COMPACT = false>
TC_HD void tc_polyline_setup(int W, int H, int32_t x0, int32_t y0, int32_t x1, int32_t y1, int t, int role, TcPrim *out) {
    int64_t ax = x0, ay = y0, bx = x1, by = y1;
    if (t <= 1) {
        if (role == TC_ROLE_ALL || role == TC_ROLE_SPANS) tc_setup_bresenham(W, H, ax, ay, bx, by, out);
        return;
    }
    ax += t; ay += t; bx += t; by += t;
    if (!tc_clip_line((int64_t)W + 2 * t, (int64_t)H + 2 * t, ax, ay, bx, by)) return;
    ax -= t; ay -= t; bx -= t; by -= t;
    int64_t P0x = ax << TC_XY_SHIFT, P0y = ay << TC_XY_SHIFT, P1x = bx << TC_XY_SHIFT, P1y = by << TC_XY_SHIFT;
    int64_t T = (int64_t)t << (TC_XY_SHIFT - 1);
    if (role != TC_ROLE_CAPS) {
        const double INV = 1.0 / TC_XY_ONE;
        double dx = (double)(P0x - P1x) * INV, dy = (double)(P1y - P0y) * INV;
        double r = dx * dx + dy * dy;
        int odd = t & 1;
        if (fabs(r) > 2.220446049250313e-16) {
            r = ((double)T + odd * TC_XY_ONE * 0.5) / sqrt(r);
            int64_t dpx = tc_cv_round(dy * r), dpy = tc_cv_round(dx * r);
            int64_t v[4][2] = {{P0x + dpx, P0y + dpy}, {P0x - dpx, P0y - dpy}, {P1x - dpx, P1y - dpy}, {P1x + dpx, P1y + dpy}};
            tc_setup_fill_convex_poly4<COMPACT>(W, H, v, role, out);
        }
    }
    if (role == TC_ROLE_ALL || role == TC_ROLE_CAPS) {
        int rad = (int)((T + (TC_XY_ONE >> 1)) >> TC_XY_SHIFT);
        for (int e = 0; e < 2; e++) {
            TcPrim &q = out[TC_SLOT_CAP0 + e];
            q.kind = TC_PRIM_CIRCLE;
            q.a[0] = (int32_t)(((e ? P1x : P0x) + (TC_XY_ONE >> 1)) >> TC_XY_SHIFT);
            q.a[1] = (int32_t)(((e ? P1y : P0y) + (TC_XY_ONE >> 1)) >> TC_XY_SHIFT);
            q.a[2] = rad;
            q.a[3] = q.a[4] = q.a[5] = q.a[6] = 0;
        }
    }
}

// 32-bit pixel helpers (coordinates are frame-sized here)
TC_HD void tc_put32(const TcPlane &pl, int x, int y) {
    if ((unsigned)x >= (unsigned)pl.W || y < pl.y_lo || y >= pl.y_hi) return;
    int b = (y - pl.row_base) * pl.W + x;
    tc_or_word(pl.bits + (b >> 5), 1u << (b & 31));
}

// filled midpoint circle; the (radius+1)-step outer loop is replayed by every lane, the 4 spans of a step go to 4 lanes
TC_HD void tc_circle_filled(const TcLanes &g, const TcPlane &pl, int cx, int cy, int radius) {
    int err = 0, dx = radius, dy = 0, plus = 1, minus = (radius << 1) - 1;
    int it = 0;
    while (dx >= dy) {
        int y11 = cy - dy, y12 = cy + dy, y21 = cy - dx, y22 = cy + dx;
        int x11 = cx - dx, x12 = cx + dx, x21 = cx - dy, x22 = cx + dy;
        if (x11 < pl.W && x12 >= 0 && y21 < pl.H && y22 >= 0) {
            if (x11 < 0) x11 = 0;
            if (x12 > pl.W - 1) x12 = pl.W - 1;
            int sub = (g.lane + g.n - (it * 4) % g.n) % g.n; // rotate the work over the lanes
            if ((g.n == 1 || sub == 0) && (unsigned)y11 < (unsigned)pl.H) tc_hline(pl, y11, x11, x12);
            if ((g.n == 1 || sub == 1) && (unsigned)y12 < (unsigned)pl.H) tc_hline(pl, y12, x11, x12);
            if (x21 < pl.W && x22 >= 0) {
                if (x21 < 0) x21 = 0;
                if (x22 > pl.W - 1) x22 = pl.W - 1;
                if ((g.n == 1 || sub == 2) && (unsigned)y21 < (unsigned)pl.H) tc_hline(pl, y21, x21, x22);
                if ((g.n == 1 || sub == 3) && (unsigned)y22 < (unsigned)pl.H) tc_hline(pl, y22, x21, x22);
            }
        }
        dy++;
        err += plus;
        plus += 2;
        int mask = (err <= 0) - 1;
        err -= minus & mask;
        dx += mask;
        minus -= mask & 2;
        it++;
    }
}

// draws one primitive with the lanes of the group
TC_HD void tc_prim_draw(const TcLanes &g, const TcPlane &pl, const TcPrim &q) {
    if (q.kind == TC_PRIM_LINE2) {
        const int base = q.a[1], fix = q.a[2], step = q.a[3], n = q.a[4];
        if (g.lane == 0) tc_put32(pl, q.a[5], q.a[6]);
        if (q.a[0]) for (int i = g.lane; i <= n; i += g.n) tc_put32(pl, base + i, (fix + i * step) >> TC_XY_SHIFT);
        else for (int i = g.lane; i <= n; i += g.n) tc_put32(pl, (fix + i * step) >> TC_XY_SHIFT, base + i);
    } else if (q.kind == TC_PRIM_SPAN) {
        const int y = q.a[0];
        int r0 = q.a[1] > pl.y_lo ? q.a[1] : pl.y_lo;
        int r1 = q.a[2] < pl.y_hi ? q.a[2] : pl.y_hi;
        for (int r = r0 + g.lane; r < r1; r += g.n) {
            int xa = q.a[3] + (r - y) * q.a[4], xb = q.a[5] + (r - y) * q.a[6];
            int xl = xa > xb ? xb : xa, xr = xa > xb ? xa : xb;
            int xx1 = (xl + (TC_XY_ONE >> 1)) >> TC_XY_SHIFT, xx2 = (xr + (TC_XY_ONE >> 1)) >> TC_XY_SHIFT;
            if (xx2 >= 0 && xx1 < pl.W) {
                if (xx1 < 0) xx1 = 0;
                if (xx2 >= pl.W) xx2 = pl.W - 1;
                tc_hline(pl, r, xx1, xx2);
            }
        }
    } else if (q.kind == TC_PRIM_CIRCLE) {
        tc_circle_filled(g, pl, q.a[0], q.a[1], q.a[2]);
    } else if (q.kind == TC_PRIM_BRES) {
        const int vert = q.a[0], x1 = q.a[1], y1 = q.a[2], sy = q.a[3];
        const unsigned dx = (unsigned)q.a[4], dy = (unsigned)q.a[5];
        if (dx == 0) {
            if (g.lane == 0) tc_put32(pl, x1, y1);
            return;
        }
        for (unsigned i = g.lane; i <= dx; i += g.n) {
            // 2*dy*i + dx - 1 < 2^32 for frame-sized lines (dx, dy < 2^15)
            int c = (int)((2u * dy * i + dx - 1u) / (2u * dx));
            if (vert) tc_put32(pl, x1 + c, y1 + sy * (int)i);
            else tc_put32(pl, x1 + (int)i, y1 + sy * c);
        }
    }
}

// setup + draw by one group (every lane replays the scalar setup); the fused kernel splits the two phases instead
TC_HD void tc_polyline2(const TcLanes &g, const TcPlane &pl, int32_t x0, int32_t y0, int32_t x1, int32_t y1, int t) {
    TcPrim prims[TC_MAX_PRIMS_PER_SEG];
    for (int i = 0; i < TC_MAX_PRIMS_PER_SEG; i++) prims[i].kind = TC_PRIM_NONE;
    tc_polyline_setup(pl.W, pl.H, x0, y0, x1, y1, t, TC_ROLE_ALL, prims);
    for (int i = 0; i < TC_MAX_PRIMS_PER_SEG; i++)
        if (prims[i].kind != TC_PRIM_NONE) tc_prim_draw(g, pl, prims[i]);
}

// ------------------------------------------------------------------------------------------------ bird's-eye view
// The BEV contract (include/tinycarlo_b200.h, tc_set_bev): a map point -> BEV pixel, float64 in the contract's order (the
// library is built without FMA contraction), truncated like np.int32
TC_HD void tc_bev_point(double x, double y, double c, double s, double k, double col0, double row0, double px, double py, int32_t &u,
                        int32_t &v) {
    const double dx = px - x, dy = py - y;
    u = tc_np_int32(col0 + k * (dy * c - dx * s));
    v = tc_np_int32(row0 - k * (dx * c + dy * s));
}

struct TcBevGeom {
    double k, col0, row0;
    int H, W, thickness, route;
};

// BEV segment i of one env: laneline edges 0..sumE-1 in table order (plane = their class), then - route on - the local-path
// edges sumE..sumE+3 (plane C). Returns false when there is no such segment or when cv2.polylines provably draws nothing for
// it: both endpoints lie beyond the same side of the frame grown by t+1 pixels (a thick line reaches at most (t+1)/2 + 1
// pixels beyond the segment between its endpoints).
TC_HD bool tc_bev_segment(const TcTrackTables &tt, const TcBevGeom &g, double x, double y, double c, double s, const int32_t *si, int i,
                          int32_t (&p)[4], int &plane) {
    const int C = tt.n_classes, sumE = tt.ll_edge_off[C];
    double ax, ay, bx, by;
    if (i < sumE) {
        int cls = 0;
        while (i >= tt.ll_edge_off[cls + 1]) cls++;
        const double *nodes = tt.ll_nodes + 2 * tt.ll_node_off[cls];
        const int32_t n0 = tt.ll_edges[2 * i], n1 = tt.ll_edges[2 * i + 1];
        ax = nodes[2 * n0]; ay = nodes[2 * n0 + 1]; bx = nodes[2 * n1]; by = nodes[2 * n1 + 1];
        plane = cls;
    } else {
        const int j = i - sumE;
        if (!g.route || j >= 4 || j >= si[TC_SI_PATH_LEN]) return false;
        const int32_t n0 = si[TC_SI_PATH_NODES + 2 * j], n1 = si[TC_SI_PATH_NODES + 2 * j + 1];
        if (n0 < 0 || n0 >= tt.lp_n_nodes || n1 < 0 || n1 >= tt.lp_n_nodes) return false;
        ax = tt.lp_nodes[2 * n0]; ay = tt.lp_nodes[2 * n0 + 1]; bx = tt.lp_nodes[2 * n1]; by = tt.lp_nodes[2 * n1 + 1];
        plane = C;
    }
    tc_bev_point(x, y, c, s, g.k, g.col0, g.row0, ax, ay, p[0], p[1]);
    tc_bev_point(x, y, c, s, g.k, g.col0, g.row0, bx, by, p[2], p[3]);
    const int64_t m = g.thickness + 1, r = (int64_t)g.W - 1 + m, b = (int64_t)g.H - 1 + m;
    return !((p[0] < -m && p[2] < -m) || (p[1] < -m && p[3] < -m) || (p[0] > r && p[2] > r) || (p[1] > b && p[3] > b));
}

// ------------------------------------------------------------------------------------------------ range scan
// The range-scan contract (include/tinycarlo_b200.h, tc_set_lidar), float64 in the contract's order (no FMA contraction).
struct TcLidarGeom {
    int rays;
    double fov, max_range, fwd, right;
};

// origin O of the rays: (fwd, right) metres in the car frame
TC_HD void tc_lidar_origin(const TcLidarGeom &g, double x, double y, double c, double s, double &ox, double &oy) {
    ox = x + (g.fwd * c - g.right * s);
    oy = y + (g.fwd * s + g.right * c);
}
// direction of ray j from the host's (a_j, b_j) = (cos phi_j, sin phi_j)
TC_HD void tc_lidar_dir(double a, double b, double c, double s, double &dx, double &dy) {
    dx = a * c - b * s;
    dy = a * s + b * c;
}

// true when RN(n / den) is certainly < 0 (not -0.0, which counts as >= 0): opposite signs, |n| >= 2^-1000 and |den| <= 2^70 make
// |n / den| >= 2^-1070, far above the 2^-1075 below which the quotient rounds to -0.0. NaN operands are never rejected here.
TC_HD bool tc_lidar_negative(double n, double den) {
    return (n < 0) != (den < 0) && fabs(n) >= 0x1p-1000 && fabs(den) <= 0x1p70;
}
// true when RN(un / den) is certainly > 1: same signs, |den| >= 2^-1000 (the product below is not subnormal) and
// |un| > RN(|den| * (1 + 2^-20)) >= |den| * (1 + 2^-20) * (1 - 2^-53) > |den| * (1 + 2^-53): the quotient lies above the midpoint
// between 1 and its successor, so it rounds above 1. A quotient that rounds to exactly 1.0 is never rejected.
TC_HD bool tc_lidar_above_one(double un, double den) {
    const double ad = fabs(den);
    return (un < 0) == (den < 0) && ad >= 0x1p-1000 && fabs(un) > ad * (1.0 + 0x1p-20);
}

// one ray (dx, dy) against one staged edge (tc_lidar_stage: ex, ey, wx, wy, tn = wx*ey - wy*ex): true and t for a hit of the
// contract. The division-free rejections above only drop pairs whose quotients provably fail the contract's tests, so the
// result is the contract's bit for bit; u is divided before t, and t only for the pairs whose u passes.
TC_HD bool tc_lidar_hit(double dx, double dy, double ex, double ey, double wx, double wy, double tn, double &t) {
    const double den = dx * ey - dy * ex;
    if (den == 0) return false;
    const double un = wx * dy - wy * dx;
    if (tc_lidar_negative(tn, den) || tc_lidar_negative(un, den) || tc_lidar_above_one(un, den)) return false;
    const double u = un / den;
    if (!(u >= 0 && u <= 1)) return false;
    t = tn / den;
    return t >= 0;
}

// Stages edge (A, B) for origin O and heading (c, s): st = {ex, ey, wx, wy, tn}. Returns false when no ray of the fan can hit
// the edge with t <= max_range (the cull), true otherwise. Conservative, including rounding:
//  - kept: every edge whose bounding box meets the square of half-size M = max_range * (1 + 2^-10) + 2^-50 * (|ox| + |oy|)
//    around O. The rounding of ox +- M costs less than 2^-51 * (M + |ox| + |oy|), so the square tested contains the one of
//    half-size max_range * (1 + 2^-11) whatever the origin's magnitude.
//  - an edge outside that square needs, for a hit with t <= max_range, the computed intersection t*d (|d| = 1 within a few
//    ulp) to be more than g = max_range * 2^-12 from the edge point A + u*e. Write z = (A + u*e - O) - t*d. The rounding of
//    den, tn, un and of the two divisions bounds |cross(z, d)| by ~5 * 2^-53 * (|w| + |e|) and |cross(z, e)| by
//    ~5 * 2^-53 * |e| * (|w| + max_range) (exact identities: cross(w, e) = t*den, cross(w, d) = u*den). With |z| >= g,
//    the component of z along d is >= g / 2, so the sine of the angle between the edge and the ray is at most
//    tol = 2^-34 * (2|w| + max_range + |e|) / max_range (16x that bound), and O lies within max_range + 2^-48 * (|w| +
//    max_range) of the edge's line. Such an edge - far away, and parallel to a ray to within tol - is kept; every other
//    edge outside the square is dropped. The 1-norms below bound the 2-norms from above.
//  - zero-length edges (den == 0 for every ray) are dropped; non-finite or huge / tiny magnitudes are kept.
TC_HD bool tc_lidar_stage(const TcLidarGeom &g, double ox, double oy, double c, double s, double ax, double ay, double bx, double by,
                          double *st) {
    const double ex = bx - ax, ey = by - ay, wx = ax - ox, wy = ay - oy;
    const double tn = wx * ey - wy * ex;
    st[0] = ex; st[1] = ey; st[2] = wx; st[3] = wy; st[4] = tn;
    const double R = g.max_range, M = R * (1.0 + 0x1p-10) + 0x1p-50 * (fabs(ox) + fabs(oy));
    const double x0 = ax < bx ? ax : bx, x1 = ax < bx ? bx : ax, y0 = ay < by ? ay : by, y1 = ay < by ? by : ay;
    if (x0 <= ox + M && x1 >= ox - M && y0 <= oy + M && y1 >= oy - M) return true;
    if (ex == 0 && ey == 0) return false;
    const double w1 = fabs(wx) + fabs(wy), e1 = fabs(ex) + fabs(ey);
    if (!(w1 <= 0x1p400 && e1 <= 0x1p400 && e1 >= 0x1p-400 && R >= 0x1p-400 && R <= 0x1p400)) return true;   // also NaN
    if (fabs(tn) > (R * (1.0 + 0x1p-40) + 0x1p-48 * (w1 + R + e1)) * e1 * (1.0 + 0x1p-40)) return false;   // line too far from O
    const double tol = 0x1p-34 * (2.0 * w1 + R + e1) / R;
    if (tol >= 0.25) return true;
    // angle of the edge in the car frame against the ray angles phi_j, lines taken modulo 180 degrees
    const double psi = atan2(ey * c - ex * s, ex * c + ey * s) * (180.0 / TC_PI);
    const double slack = (2.0 * tol + 0x1p-40) * (180.0 / TC_PI);
    for (int k = -2; k <= 2; k++) {
        const double a = psi + 180.0 * k;
        double j = rint((a + g.fov / 2) / g.fov * g.rays - 0.5);
        j = j < 0 ? 0 : (j > g.rays - 1 ? g.rays - 1 : j);
        if (fabs(a - (g.fov * ((j + 0.5) / g.rays) - g.fov / 2)) <= slack) return true;
    }
    return false;
}
