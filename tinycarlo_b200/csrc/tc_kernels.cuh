// tc_kernels.cuh — sm_100a kernels of the hot path. Included by tc_api.cu only.
//
//   tc_track_kernel              a warp per env: bicycle step, local-path selection, CTE / heading / laneline distances
//                                (nearest-laneline index), reward, flags, pose for the camera, resets with device-side spawn
//                                draws. Map tables are staged once per block into shared memory with a 1-D TMA bulk copy
//                                (cp.async.bulk + mbarrier) and shared by the block's 8 envs.
//   tc_render_classes_kernel     THE HEADLINE KERNEL (large u8 / bf16 / bit frames): a block per (env, class) - camera pass,
//                                polyline set-up, drawing into a 1-bit plane in shared memory, bits -> bytes with 128-bit
//                                streaming stores; every output byte is written exactly once. Runs at the HBM write ceiling.
//   tc_render_env_kernel         small frames: a block per env renders all classes, camera pass on the visible-set
//                                sub-graph of the camera's ground cell, one thread per primitive.
//   tc_render_env_banded_kernel  large RGB / bit-packed frames: a block per env, set-up once, row bands inside the block.
//   tc_project_kernel + tc_raster_classes_kernel / tc_raster_rgb_kernel
//                                the unfused fallback (segments through global memory, a block per row band) and the
//                                debug segment export.
//   tc_noise_blobs_kernel        NoiseObservationWrapper; tc_debug_layer_kernel: layer.py known-answer hook for the tests.
#pragma once
#include <cuda_runtime.h>

#include "tc_core.cuh"

#define TC_TRACK_THREADS 256
#define TC_PROJ_THREADS 128
#define TC_RASTER_THREADS 256
#define TC_SETUP_CHUNK 16 // segments set up per round (one thread per segment and role), then drawn by all warps
#define TC_ENV_SEG_WORDS (12 * 8 + 1) // block-per-env kernels: a segment's 12 primitive slots of 8 words, padded so that lanes reading one slot of 32 segments hit 32 banks

// ------------------------------------------------------------------------------------------------ TMA / mbarrier PTX
__device__ __forceinline__ uint32_t tc_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void tc_fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc_smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(tc_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(uint64_t *bar, uint32_t phase) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(tc_smem_u32(bar)),
        "r"(phase)
        : "memory");
}
// 128-bit streaming store (evict-first: the observation is consumed by a later kernel, never re-read here)
__device__ __forceinline__ void tc_st_cs(void *p, uint4 v) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// ------------------------------------------------------------------------------------------------ tracking
struct TcTrackArgs {
    const unsigned char *blob; // packed map tables (global)
    TcBlobLayout layout;
    int n_envs;
    int n_cams;   // M cameras per env: view v = env * M + m
    int mode;     // 0 = step, 1 = reset
    int wrapped;
    double *sf;
    int32_t *si;
    const double *car;   // [N, TC_CP_N]
    const double *cam;   // [N*M, TC_CAM_N]
    double *pose;        // [N*M, 12] out
    const float *act_cc; // [N,2]
    const double *act_cc64; // [N,2] optional float64 actions (single-env drop-in: Python-float actions keep full precision)
    const int32_t *act_man;
    const uint8_t *mask;        // reset: envs to reset (NULL = all)
    uint8_t *view_mask;         // reset, optional [N*M] out: mask[env] for each of the env's views (the render kernels index masks by view)
    const int32_t *spawn_nodes; // reset
    // next-step autoreset (gymnasium AutoresetMode.NEXT_STEP): an env whose previous step ended is reset by this step
    uint8_t *done;              // [N] in/out, NULL = autoreset off
    uint8_t *was_reset;         // [N] out, optional: 1 when this step reset the env instead of stepping it
    // spawn draws on the device (tc_set_spawn_rng): per-env PCG64 state, optional spawn_points list, last node drawn
    uint64_t *rng;              // [N, TC_RNG_N]
    const int32_t *spawn_points;
    int n_spawn_points;
    int32_t *last_spawn;        // [N] out: lanepath node of the env's most recent reset
    // nearest-laneline index (global memory; near_nx == 0: none)
    double near_x0, near_y0, near_inv_cell;
    int near_nx, near_ny;
    const int32_t *near_off;
    const uint16_t *near_edge;
    TcOutputs out;
};

// The end of a tracking step, shared by both tracking kernels (one thread per env calls it): autoreset flags, state, the pose for
// the camera pass and the outputs the caller asked for.
__device__ __forceinline__ void tc_track_store(const TcTrackArgs &a, const TcTrackTables &t, int env, double *sf, int32_t *si, const TcCarState &s,
                                               const TcInfo &info, bool truncated, bool auto_reset, const double *dist, const int *nearest) {
    const int C = t.n_classes;
    if (a.mode == 0 && a.done) a.done[env] = (info.terminated || truncated) ? 1 : 0;
    if (a.mode == 0 && a.was_reset) a.was_reset[env] = auto_reset ? 1 : 0;
    tc_store_state(sf, si, s);
    // poses of the env's M views for the camera pass: front-axle update already evaluated cos/sin(rot); recomputing keeps the code simple
    {
        const double c = cos(s.rot), sn = sin(s.rot);
        for (int m = 0; m < a.n_cams; m++) {
            const size_t v = (size_t)env * a.n_cams + m;
            tc_camera_pose(a.cam + v * TC_CAM_N + TC_CAM_E, s.x, s.y, c, sn, a.pose + v * 12);
        }
    }
    const TcOutputs &o = a.out;
    if (o.cte) o.cte[env] = (float)info.cte;
    if (o.heading_error) o.heading_error[env] = (float)info.heading;
    if (o.velocity) o.velocity[env] = (float)info.velocity;
    if (o.position) { o.position[2 * env] = (float)s.x; o.position[2 * env + 1] = (float)s.y; }
    if (o.orientation) o.orientation[env] = (float)s.rot;
    if (o.laneline_distances) for (int c = 0; c < C; c++) o.laneline_distances[(size_t)env * C + c] = (float)dist[c];
    if (o.nearest_edge) for (int c = 0; c < C; c++) o.nearest_edge[(size_t)env * C + c] = nearest[c];
    // car.py:66 builds local_path coordinates only when the info is non-empty (len >= 2)
    int plen = s.path_len >= 2 ? s.path_len : 0;
    if (o.local_path)
        for (int i = 0; i < 4; i++) {
            bool ok = i < plen;
            o.local_path[(size_t)env * 8 + 2 * i] = ok ? (float)t.lp_nodes[2 * s.pn[2 * i + 1]] : 0.0f;
            o.local_path[(size_t)env * 8 + 2 * i + 1] = ok ? (float)t.lp_nodes[2 * s.pn[2 * i + 1] + 1] : 0.0f;
        }
    if (o.local_path_nodes)
        for (int i = 0; i < 8; i++) o.local_path_nodes[(size_t)env * 8 + i] = (i >> 1) < s.path_len ? s.pn[i] : -1;
    if (o.path_len) o.path_len[env] = s.path_len;
    if (o.info_f64) {
        double *r = o.info_f64 + (size_t)env * (4 + C);
        r[TC_INFO_CTE] = info.cte; r[TC_INFO_HEADING] = info.heading; r[TC_INFO_VELOCITY] = info.velocity;
        if (a.mode == 0) r[TC_INFO_REWARD] = info.reward;
        for (int c = 0; c < C; c++) r[TC_INFO_DIST0 + c] = dist[c];
    }
    if (a.mode == 0) {
        if (o.reward) o.reward[env] = (float)info.reward;
        if (o.terminated) o.terminated[env] = info.terminated ? 1 : 0;
        if (o.truncated) o.truncated[env] = truncated ? 1 : 0;
    }
}

// Reset mode with a camera rig: the caller's mask value of the env for each of its views (a.view_mask is set only together with
// a.mask). Written before the reset can return early, so that a selected env whose reset fails is rendered at its old pose.
__device__ __forceinline__ void tc_store_view_mask(const TcTrackArgs &a, int env) {
    for (int m = 0; m < a.n_cams; m++) a.view_mask[(size_t)env * a.n_cams + m] = a.mask[env];
}

// G lanes per env (a power of two <= 32): the scalar part of a step is computed redundantly by the G lanes, the scans are spread
// over them. 32 = a warp per env; 8 = four envs per warp, a quarter of the warps for the same envs - the better choice when a few
// thousand envs cannot fill the SMs with one thread each (4096 envs: 1024 instead of 4096 warps, one wave instead of two).
template <int G>
__global__ void __launch_bounds__(TC_TRACK_THREADS, 3) tc_track_kernel(const TcTrackArgs a) {
    extern __shared__ __align__(128) unsigned char smem_blob[];
    __shared__ __align__(8) uint64_t bar;
    if (threadIdx.x == 0) {
        tc_mbar_init(&bar, 1);
        tc_fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        tc_mbar_expect_tx(&bar, (uint32_t)a.layout.total_bytes);
        tc_bulk_g2s(smem_blob, a.blob, (uint32_t)a.layout.total_bytes, &bar);
    }
    const int env = blockIdx.x * (TC_TRACK_THREADS / G) + (int)threadIdx.x / G;
    TcLanes g = {(int)(threadIdx.x & (G - 1)), G};
    const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) & ~(G - 1)));   // the lanes of this env's group
    const int leader = (threadIdx.x & 31) & ~(G - 1);
    tc_mbar_wait(&bar, 0);
    if (env >= a.n_envs) return;
    TcTrackTables t = tc_track_tables(smem_blob, a.layout);
    t.near_x0 = a.near_x0; t.near_y0 = a.near_y0; t.near_inv_cell = a.near_inv_cell; t.near_nx = a.near_nx; t.near_ny = a.near_ny;
    t.near_off = a.near_off; t.near_edge = a.near_edge;
    const double *cp = a.car + (size_t)env * TC_CP_N;
    double *sf = a.sf + (size_t)env * TC_SF_N;
    int32_t *si = a.si + (size_t)env * TC_SI_N;
    TcCarState s;
    bool truncated = false;
    bool auto_reset = false;
    if (a.mode == 0 && a.done && a.done[env]) {
        // the action of this step is ignored; reward 0, not terminated, not truncated, empty info (env.py:101-113)
        int node = -1;
        if (g.lane == 0 && a.rng) node = tc_spawn_draw(t, a.rng + (size_t)env * TC_RNG_N, a.spawn_points, a.n_spawn_points);
        node = __shfl_sync(gmask, node, leader);
        tc_load_state(sf, si, s);
        auto_reset = tc_car_reset(t, cp, s, node);
        if (auto_reset && g.lane == 0 && a.last_spawn) a.last_spawn[env] = node;
    }
    if (auto_reset) {
    } else if (a.mode == 1) {
        if (a.view_mask && g.lane == 0) tc_store_view_mask(a, env);
        if (a.mask && !a.mask[env]) return;
        tc_load_state(sf, si, s);
        int node = -1;
        if (a.spawn_nodes) node = a.spawn_nodes[env];
        else {
            if (g.lane == 0 && a.rng) node = tc_spawn_draw(t, a.rng + (size_t)env * TC_RNG_N, a.spawn_points, a.n_spawn_points);
            node = __shfl_sync(gmask, node, leader);
        }
        if (!tc_car_reset(t, cp, s, node)) return;
        if (g.lane == 0 && a.last_spawn) a.last_spawn[env] = node;
    } else {
        tc_load_state(sf, si, s);
        // env.py:118: np.clip(action["car_control"], -1, 1) on float64
        double v_raw = a.act_cc64 ? a.act_cc64[2 * env] : (double)a.act_cc[2 * env];
        double s_raw = a.act_cc64 ? a.act_cc64[2 * env + 1] : (double)a.act_cc[2 * env + 1];
        double v_cmd = tc_np_clip(v_raw, -1.0, 1.0), s_cmd = tc_np_clip(s_raw, -1.0, 1.0);
        truncated = tc_car_step(g, t, cp, s, v_cmd, s_cmd, a.act_man[env]);
    }
    double dist[TC_MAX_CLASSES];
    int nearest[TC_MAX_CLASSES];
    TcInfo info = tc_get_info(g, t, cp, s, a.wrapped != 0, dist, nearest);
    if (auto_reset) { info.reward = 0; info.terminated = false; }
    if (g.lane != 0) return;
    tc_track_store(a, t, env, sf, si, s, info, truncated, auto_reset, dist, nearest);
}

// The same step with ONE THREAD PER ENV. The warp-per-env kernel above computes the scalar part of a step (bicycle model, path
// hops, distances) redundantly in all 32 lanes and only spreads the two scans; since the nearest-laneline index went in, those
// scans are a handful of candidates long, so almost all of its issue slots are redundant work. Here every thread owns an env;
// the two O(E) scans that remain - the u-turn's global search (car.py:130-131) and the laneline search of a car outside the
// index grid - are run by the whole warp on behalf of each lane that needs one (ballot loop), with the same lexicographic
// arg-min, so results are bit-identical to the kernel above. 32x fewer warps for the same envs: 0.19 -> 0.03 ms for 32768 envs.
#define TC_TRACK1_THREADS 128
__global__ void __launch_bounds__(TC_TRACK1_THREADS) tc_track_thread_kernel(const TcTrackArgs a) {
    extern __shared__ __align__(128) unsigned char smem_blob[];
    __shared__ __align__(8) uint64_t bar;
    if (threadIdx.x == 0) {
        tc_mbar_init(&bar, 1);
        tc_fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        tc_mbar_expect_tx(&bar, (uint32_t)a.layout.total_bytes);
        tc_bulk_g2s(smem_blob, a.blob, (uint32_t)a.layout.total_bytes, &bar);
    }
    const int lane = threadIdx.x & 31;
    const int env_raw = blockIdx.x * TC_TRACK1_THREADS + threadIdx.x;
    const bool in_range = env_raw < a.n_envs;
    const int env = in_range ? env_raw : a.n_envs - 1;   // idle lanes shadow the last env (they take part in the warp scans) and store nothing
    const TcLanes g1 = {0, 1}, gw = {lane, 32};
    tc_mbar_wait(&bar, 0);
    TcTrackTables t = tc_track_tables(smem_blob, a.layout);
    t.near_x0 = a.near_x0; t.near_y0 = a.near_y0; t.near_inv_cell = a.near_inv_cell; t.near_nx = a.near_nx; t.near_ny = a.near_ny;
    t.near_off = a.near_off; t.near_edge = a.near_edge;
    const int C = t.n_classes;
    const double *cp = a.car + (size_t)env * TC_CP_N;
    double *sf = a.sf + (size_t)env * TC_SF_N;
    int32_t *si = a.si + (size_t)env * TC_SI_N;
    TcCarState s;
    tc_load_state(sf, si, s);
    bool truncated = false, auto_reset = false, live = in_range;   // live: this thread's env takes part in this launch
    int man = 0;
    bool stepping = false;
    if (a.mode == 0 && a.done && a.done[env]) {
        // the action of this step is ignored; reward 0, not terminated, not truncated, empty info (env.py:101-113)
        int node = -1;
        if (a.rng && in_range) node = tc_spawn_draw(t, a.rng + (size_t)env * TC_RNG_N, a.spawn_points, a.n_spawn_points);
        auto_reset = tc_car_reset(t, cp, s, node);
        if (auto_reset && in_range && a.last_spawn) a.last_spawn[env] = node;
    }
    if (auto_reset) {
    } else if (a.mode == 1) {
        if (a.view_mask && in_range) tc_store_view_mask(a, env);
        if (a.mask && !a.mask[env]) live = false;
        else {
            int node = -1;
            if (a.spawn_nodes) node = a.spawn_nodes[env];
            else if (a.rng && in_range) node = tc_spawn_draw(t, a.rng + (size_t)env * TC_RNG_N, a.spawn_points, a.n_spawn_points);
            if (!tc_car_reset(t, cp, s, node)) live = false;
            else if (in_range && a.last_spawn) a.last_spawn[env] = node;
        }
    } else {
        // env.py:118: np.clip(action["car_control"], -1, 1) on float64
        double v_raw = a.act_cc64 ? a.act_cc64[2 * env] : (double)a.act_cc[2 * env];
        double s_raw = a.act_cc64 ? a.act_cc64[2 * env + 1] : (double)a.act_cc[2 * env + 1];
        man = a.act_man[env];
        tc_car_move(cp, s, tc_np_clip(v_raw, -1.0, 1.0), tc_np_clip(s_raw, -1.0, 1.0));
        stepping = in_range;
    }
    // ---- warp-cooperative part 1: the u-turn's global edge search for the lanes that start one
    int uturn_edge = -1;
    {
        const bool want = stepping && tc_wants_uturn_scan(t, s, man);
        const double dir = want ? tc_uturn_direction(t, s, man) : 0.0;
        for (unsigned mk = __ballot_sync(0xffffffffu, want); mk; mk &= mk - 1) {
            const int src = __ffs(mk) - 1;
            const double fx = __shfl_sync(0xffffffffu, s.fx, src), fy = __shfl_sync(0xffffffffu, s.fy, src), d = __shfl_sync(0xffffffffu, dir, src);
            const int e = tc_uturn_scan(gw, t, fx, fy, d);
            if (lane == src) uturn_edge = e;
        }
    }
    if (stepping) truncated = tc_find_local_path_given(t, s, man, uturn_edge);
    // ---- warp-cooperative part 2: laneline search over all edges for cars outside the nearest-laneline index
    int pre[TC_MAX_CLASSES];
    const bool scan = live && s.path_len >= 2 && tc_near_cell(t, s.x, s.y) < 0;
    for (unsigned mk = __ballot_sync(0xffffffffu, scan); mk; mk &= mk - 1) {
        const int src = __ffs(mk) - 1;
        const double x = __shfl_sync(0xffffffffu, s.x, src), y = __shfl_sync(0xffffffffu, s.y, src);
        for (int c = 0; c < C; c++) {
            const int e = tc_nearest_laneline_scan(gw, t, c, x, y);
            if (lane == src) pre[c] = e;
        }
    }
    if (!live) return;
    double dist[TC_MAX_CLASSES];
    int nearest[TC_MAX_CLASSES];
    TcInfo info = tc_get_info(g1, t, cp, s, a.wrapped != 0, dist, nearest, scan ? pre : nullptr);
    if (auto_reset) { info.reward = 0; info.terminated = false; }
    tc_track_store(a, t, env, sf, si, s, info, truncated, auto_reset, dist, nearest);
}

// ------------------------------------------------------------------------------------------------ camera pass
struct TcProjArgs {
    const TcClassTables *classes; // [C] device array
    int n_envs, n_classes, sum_edges, max_nodes;
    int H, W;
    const int32_t *edge_off; // [C+1] device
    const double *pose;      // [N,12]
    const double *cam;       // [N,TC_CAM_N]
    const uint8_t *mask;     // optional
    int32_t *seg;            // [N, sumE, 4]
    int32_t *seg_count;      // [N, C]
};

__host__ __device__ inline size_t tc_proj_smem_bytes(int max_nodes) {
    size_t n = (size_t)((max_nodes + 15) & ~15);
    return n * (3 * sizeof(double) + 2 * sizeof(int32_t) + 5);
}

__global__ void __launch_bounds__(TC_PROJ_THREADS) tc_project_kernel(const TcProjArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int warp_cnt[TC_PROJ_THREADS / 32];
    __shared__ int base_cnt;
    const int env = blockIdx.x / a.n_classes, c = blockIdx.x % a.n_classes;
    if (a.mask && !a.mask[env]) return;
    const TcClassTables ct = a.classes[c];
    const int n = ct.n_nodes, m = ct.n_edges;
    const size_t np = (size_t)((a.max_nodes + 15) & ~15);
    TcProjScratch sc;
    sc.Px = (double *)smem_raw; sc.Py = sc.Px + np; sc.Pz = sc.Py + np;
    sc.ix = (int32_t *)(sc.Pz + np); sc.iy = sc.ix + np;
    uint8_t *fA = (uint8_t *)(sc.iy + np), *fB = fA + np, *rA = fB + np, *rB = rA + np;
    sc.vis = rB + np;
    sc.front = fA; sc.inr = rA;
    const int tid = threadIdx.x;
    double pose[12], cam[TC_CAM_N];
#pragma unroll
    for (int i = 0; i < 12; i++) pose[i] = a.pose[(size_t)env * 12 + i];
#pragma unroll
    for (int i = TC_CAM_FX; i <= TC_CAM_MAX_RANGE; i++) cam[i] = a.cam[(size_t)env * TC_CAM_N + i];
    const double max_range = cam[TC_CAM_MAX_RANGE];

    for (int v = tid; v < n; v += TC_PROJ_THREADS) {
        double X, Y, Z;
        tc_transform_node(pose, ct.nodes[2 * v], ct.nodes[2 * v + 1], X, Y, Z);
        sc.Px[v] = X; sc.Py[v] = Y; sc.Pz[v] = Z;
        fA[v] = Z < 0;
    }
    __syncthreads();
    // camera.py:70-77 near-plane fix-ups
    for (int v = tid; v < n; v += TC_PROJ_THREADS) fB[v] = fA[v] | (uint8_t)tc_clip_pass_node(ct, sc, fA, v, true, -0.0000001);
    __syncthreads();
    for (int v = tid; v < n; v += TC_PROJ_THREADS) fA[v] = fB[v] | (uint8_t)tc_clip_pass_node(ct, sc, fB, v, false, -0.0000001);
    __syncthreads();
    // camera.py:80-86 range fix-ups (depths is a live view: evaluated on the moved z)
    for (int v = tid; v < n; v += TC_PROJ_THREADS) rA[v] = sc.Pz[v] > -max_range;
    __syncthreads();
    for (int v = tid; v < n; v += TC_PROJ_THREADS) rB[v] = rA[v] | (uint8_t)tc_clip_pass_node(ct, sc, rA, v, true, -max_range);
    __syncthreads();
    for (int v = tid; v < n; v += TC_PROJ_THREADS) rA[v] = rB[v] | (uint8_t)tc_clip_pass_node(ct, sc, rB, v, false, -max_range);
    __syncthreads();
    // camera.py:89-93 projection and node visibility
    for (int v = tid; v < n; v += TC_PROJ_THREADS) {
        double u, w;
        tc_project(cam, sc.Px[v], sc.Py[v], sc.Pz[v], u, w);
        sc.ix[v] = tc_np_int32(u);
        sc.iy[v] = tc_np_int32(w);
        sc.vis[v] = (u > 0 && u < a.W && w > 0 && w < a.H && fA[v] && rA[v]) ? 1 : 0;
    }
    if (tid == 0) base_cnt = 0;
    __syncthreads();
    // camera.py:95: keep edges with >= 1 visible endpoint, in edge order (ordered block compaction)
    int32_t *seg = a.seg + ((size_t)env * a.sum_edges + a.edge_off[c]) * 4;
    for (int e0 = 0; e0 < m; e0 += TC_PROJ_THREADS) {
        int e = e0 + tid;
        int n0 = 0, n1 = 0;
        bool keep = false;
        if (e < m) {
            n0 = ct.edges[2 * e]; n1 = ct.edges[2 * e + 1];
            keep = sc.vis[n0] || sc.vis[n1];
        }
        unsigned bal = __ballot_sync(0xffffffffu, keep);
        if ((tid & 31) == 0) warp_cnt[tid >> 5] = __popc(bal);
        __syncthreads();
        int pos = base_cnt + __popc(bal & ((1u << (tid & 31)) - 1));
        for (int w = 0; w < (tid >> 5); w++) pos += warp_cnt[w];
        if (keep) {
            int4 s4 = make_int4(sc.ix[n0], sc.iy[n0], sc.ix[n1], sc.iy[n1]);
            *(int4 *)(seg + 4 * pos) = s4;
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < TC_PROJ_THREADS / 32; w++) tot += warp_cnt[w];
            base_cnt += tot;
        }
        __syncthreads();
    }
    if (tid == 0) a.seg_count[(size_t)env * a.n_classes + c] = base_cnt;
}

// ------------------------------------------------------------------------------------------------ rasterise + store
struct TcRasterArgs {
    int n_envs, n_classes, sum_edges;
    int H, W;
    int rows_per_band, n_bands;
    int plane_words; // 32-bit words of one band plane (incl. one pad word)
    const int32_t *edge_off;   // [C+1] device
    const int32_t *thickness;  // [N]
    const uint8_t *mask;       // optional
    const int32_t *seg;        // [N, sumE, 4]
    const int32_t *seg_count;  // [N, C]
    uint8_t *obs;
    uint8_t colors[TC_MAX_CLASSES * 3];
};

// 16 bits of the plane starting at bit offset o (plane has a pad word, so reading word+1 is always in bounds)
__device__ __forceinline__ uint32_t tc_bits16(const uint32_t *plane, uint32_t o) {
    uint32_t w = o >> 5;
    return __funnelshift_r(plane[w], plane[w + 1], o & 31) & 0xffffu;
}
// 4 bits -> 4 bytes of 0x00 / 0xFF
__device__ __forceinline__ uint32_t tc_expand4(uint32_t b) { return (((b & 0xfu) * 0x00204081u) & 0x01010101u) * 0xffu; }
__device__ __forceinline__ uint4 tc_expand16(uint32_t b) {
    return make_uint4(tc_expand4(b), tc_expand4(b >> 4), tc_expand4(b >> 8), tc_expand4(b >> 12));
}

// Stream `nbytes` bytes of 0/255 to `out` from the bit plane (bit i <-> byte i). `any` false: plane is known empty.
template <int NT = TC_RASTER_THREADS>
__device__ __forceinline__ void tc_store_plane(uint8_t *out, size_t nbytes, const uint32_t *plane, bool any) {
    const int tid = threadIdx.x;
    size_t head = (16 - ((uintptr_t)out & 15)) & 15;
    if (head > nbytes) head = nbytes;
    for (size_t i = tid; i < head; i += NT) out[i] = (any && ((plane[i >> 5] >> (i & 31)) & 1)) ? 255 : 0;
    const size_t nvec = (nbytes - head) >> 4;
    uint4 *o4 = (uint4 *)(out + head);
    if (!any) {
        const uint4 z = make_uint4(0, 0, 0, 0);
        size_t j = tid;
        for (; j + 3 * NT < nvec; j += 4 * NT) {
            tc_st_cs(o4 + j, z);
            tc_st_cs(o4 + j + NT, z);
            tc_st_cs(o4 + j + 2 * NT, z);
            tc_st_cs(o4 + j + 3 * NT, z);
        }
        for (; j < nvec; j += NT) tc_st_cs(o4 + j, z);
    } else {
        size_t j = tid;
        for (; j + 3 * NT < nvec; j += 4 * NT) {
            uint32_t b0 = tc_bits16(plane, (uint32_t)(head + 16 * j));
            uint32_t b1 = tc_bits16(plane, (uint32_t)(head + 16 * (j + NT)));
            uint32_t b2 = tc_bits16(plane, (uint32_t)(head + 16 * (j + 2 * NT)));
            uint32_t b3 = tc_bits16(plane, (uint32_t)(head + 16 * (j + 3 * NT)));
            tc_st_cs(o4 + j, tc_expand16(b0));
            tc_st_cs(o4 + j + NT, tc_expand16(b1));
            tc_st_cs(o4 + j + 2 * NT, tc_expand16(b2));
            tc_st_cs(o4 + j + 3 * NT, tc_expand16(b3));
        }
        for (; j < nvec; j += NT) tc_st_cs(o4 + j, tc_expand16(tc_bits16(plane, (uint32_t)(head + 16 * j))));
    }
    for (size_t i = head + (nvec << 4) + tid; i < nbytes; i += NT)
        out[i] = (any && ((plane[i >> 5] >> (i & 31)) & 1)) ? 255 : 0;
}

// The same for the block-per-env kernels, whose time goes into instructions rather than into the stores: a frame is mostly
// background, so the 0x00/0xFF expansion is skipped for the (97 % of) vectors whose 16 plane bits are all clear.
// (Tried in round 2 and rejected: for aligned output, four half-word loads per thread and a warp ballot that writes 4 x 32 background
// vectors at once - the store phase falls from 37 % to ~12 % of the packed kernel's instructions, but the bursts of back-to-back
// stores made every small-frame configuration 3-4 % SLOWER: the per-vector work paces the stores.)
template <int NT>
__device__ __forceinline__ void tc_store_plane_sparse(uint8_t *out, size_t nbytes, const uint32_t *plane, bool any) {
    const int tid = threadIdx.x;
    size_t head = (16 - ((uintptr_t)out & 15)) & 15;
    if (head > nbytes) head = nbytes;
    for (size_t i = tid; i < head; i += NT) out[i] = (any && ((plane[i >> 5] >> (i & 31)) & 1)) ? 255 : 0;
    const size_t nvec = (nbytes - head) >> 4;
    uint4 *o4 = (uint4 *)(out + head);
    const uint4 z = make_uint4(0, 0, 0, 0);
    if (!any) {
        for (size_t j = tid; j < nvec; j += NT) tc_st_cs(o4 + j, z);
    } else {
        for (size_t j = tid; j < nvec; j += NT) {
            const uint32_t b = tc_bits16(plane, (uint32_t)(head + 16 * j));
            if (b == 0) tc_st_cs(o4 + j, z);
            else tc_st_cs(o4 + j, tc_expand16(b));
        }
    }
    for (size_t i = head + (nvec << 4) + tid; i < nbytes; i += NT)
        out[i] = (any && ((plane[i >> 5] >> (i & 31)) & 1)) ? 255 : 0;
}

// colour of class i as r | g<<8 | b<<16 from the kernel-parameter byte array, with compile-time indexing only: a runtime
// index makes the compiler copy the whole array into every thread's local memory at kernel entry
__device__ __forceinline__ uint32_t tc_color24_of(const uint8_t (&colors)[TC_MAX_CLASSES * 3], int i) {
    uint32_t v = 0;
#pragma unroll
    for (int k = 0; k < TC_MAX_CLASSES; k++)
        if (k == i) v = colors[3 * k] | (colors[3 * k + 1] << 8) | (colors[3 * k + 2] << 16);
    return v;
}

// RGB composition from C class planes (class c starts at bit c*stride_bits of `planes`; a pad word follows the last
// plane): byte q of the [rows,W,3] image belongs to pixel q/3, channel q%3, and takes the colour of the LAST class drawn
// there (painter's order, renderer.py:41-43). 16 output bytes touch at most 6 pixels: one funnel-shifted 6-bit window per
// class gives the winning colour of each of them; the 16 bytes are then cut out of that 18-byte pixel stream by funnel shifts.
template <int NT>
__device__ __forceinline__ void tc_store_rgb(uint8_t *out, uint32_t npx, const uint32_t *planes, uint32_t stride_bits, int C,
                                             const uint32_t *color24 /* shared: r | g<<8 | b<<16 per class */, bool any,
                                             const uint32_t *any_plane = nullptr /* optional OR of the class planes */) {
    const int tid = threadIdx.x;
    const uint32_t nbytes = npx * 3u;
    auto byte_at = [&](uint32_t q) -> uint8_t {   // scalar path for the unaligned head / tail
        if (!any) return 0;
        uint32_t p = q / 3u;
        uint32_t v = 0;
        for (int c = 0; c < C; c++) {
            uint32_t bi = (uint32_t)c * stride_bits + p;
            if ((planes[bi >> 5] >> (bi & 31)) & 1) v = color24[c];
        }
        return (uint8_t)(v >> (8 * (q - 3u * p)));
    };
    uint32_t head = (16u - (uint32_t)((uintptr_t)out & 15)) & 15u;
    if (head > nbytes) head = nbytes;
    for (uint32_t i = tid; i < head; i += NT) out[i] = byte_at(i);
    const uint32_t nvec = (nbytes - head) >> 4;
    uint4 *o4 = (uint4 *)(out + head);
    // the 16 bytes of vector j from the class planes (the caller knows, or does not care, that its window is not empty)
    auto compose = [&](uint32_t j) -> uint4 {
        const uint32_t q0 = head + 16u * j;
        const uint32_t p0 = q0 / 3u;
        // the 18-byte stream of the 6 pixels the vector touches, in five words (pixel k = bits 24k .. 24k+23); kept in scalars:
        // an indexed array would live in local memory, and its traffic queues behind the observation stores
        uint32_t s0 = 0, s1 = 0, s2 = 0, s3 = 0, s4 = 0;
        for (int c = 0; c < C; c++) {
            uint32_t bi = (uint32_t)c * stride_bits + p0;
            uint32_t w = __funnelshift_r(planes[bi >> 5], planes[(bi >> 5) + 1], bi & 31) & 0x3fu;
            if (w) {   // painter's order: a later class replaces the pixel
                const uint32_t cc = color24[c];
                if (w & 1u) s0 = (s0 & 0xff000000u) | cc;
                if (w & 2u) { s0 = (s0 & 0x00ffffffu) | (cc << 24); s1 = (s1 & 0xffff0000u) | (cc >> 8); }
                if (w & 4u) { s1 = (s1 & 0x0000ffffu) | (cc << 16); s2 = (s2 & 0xffffff00u) | (cc >> 16); }
                if (w & 8u) s2 = (s2 & 0x000000ffu) | (cc << 8);
                if (w & 16u) s3 = (s3 & 0xff000000u) | cc;
                if (w & 32u) { s3 = (s3 & 0x00ffffffu) | (cc << 24); s4 = (s4 & 0xffff0000u) | (cc >> 8); }
            }
        }
        const uint32_t sh = 8u * (q0 - 3u * p0);   // the vector starts at byte 0, 1 or 2 of the stream
        return make_uint4(__funnelshift_r(s0, s1, sh), __funnelshift_r(s1, s2, sh), __funnelshift_r(s2, s3, sh), __funnelshift_r(s3, s4, sh));
    };
    const uint4 zero = make_uint4(0, 0, 0, 0);
    if (!any) {
        for (uint32_t j = tid; j < nvec; j += NT) tc_st_cs(o4 + j, zero);
    } else if (!any_plane) {
        for (uint32_t j = tid; j < nvec; j += NT) tc_st_cs(o4 + j, compose(j));
    } else {
        // A frame is mostly background, and the few vectors that are not are scattered over the lanes of a warp: composing
        // them where they fall runs the class loop with 2-3 active lanes. So a warp writes the empty vectors at once and
        // queues the others (warp-private queue in shared memory); whenever 32 are waiting they are composed with all lanes.
        __shared__ uint32_t wq[NT / 32][64];
        const uint32_t lane = tid & 31, warp = tid >> 5;
        uint32_t qn = 0;   // warp-uniform
        auto visit = [&](uint32_t j, bool valid) {   // called by all lanes of the warp
            bool look = false;
            if (valid) {
                const uint32_t p0 = (head + 16u * j) / 3u;
                look = (__funnelshift_r(any_plane[p0 >> 5], any_plane[(p0 >> 5) + 1], p0 & 31) & 0x3fu) != 0u;
                if (!look) tc_st_cs(o4 + j, zero);
            }
            const unsigned m = __ballot_sync(0xffffffffu, look);
            if (m) {
                if (look) wq[warp][qn + __popc(m & ((1u << lane) - 1u))] = j;
                qn += __popc(m);
                __syncwarp();
                if (qn >= 32u) {
                    const uint32_t jj = wq[warp][qn - 32u + lane];
                    tc_st_cs(o4 + jj, compose(jj));
                    qn -= 32u;
                    __syncwarp();
                }
            }
        };
        uint32_t done = 0;
        if (head == 0) {
            // 32 words of the OR plane = 1024 pixels = 3072 bytes = 192 vectors: when they are all empty the warp writes its
            // 6 x 32 zero vectors without any per-vector work
            const uint32_t ngroups = nvec / 192u;
            for (uint32_t gi = warp; gi < ngroups; gi += NT / 32) {
                const unsigned nz = __ballot_sync(0xffffffffu, any_plane[gi * 32u + lane] != 0u);
                const uint32_t j0 = gi * 192u + lane;
                if (nz == 0) {
#pragma unroll
                    for (int k = 0; k < 6; k++) tc_st_cs(o4 + j0 + 32u * k, zero);
                } else {
                    for (int k = 0; k < 6; k++) visit(j0 + 32u * k, true);
                }
            }
            done = ngroups * 192u;
        }
        for (uint32_t base = done + warp * 32u; base < nvec; base += NT) visit(base + lane, base + lane < nvec);
        if (lane < qn) {
            const uint32_t jj = wq[warp][lane];
            tc_st_cs(o4 + jj, compose(jj));
        }
    }
    for (uint32_t i = head + (nvec << 4) + tid; i < nbytes; i += NT) out[i] = byte_at(i);
}

// Observation formats of the fused kernel beyond the reference's two (SURVEY 8f-1: emit what the policy consumes):
//   BITS  the bit plane itself, 1 bit per pixel (bit i of the little-endian byte stream = pixel i, i = y*W + x): 8x fewer bytes
//   BF16  0.0 / 1.0 in bfloat16 [N,C,H,W]: the u8 -> float /255 normalisation kernel of the consumer disappears
enum { TC_FMT_U8 = 0, TC_FMT_RGB = 1, TC_FMT_BITS = 2, TC_FMT_BF16 = 3 };

template <int NT>
__device__ __forceinline__ void tc_store_bits(uint32_t *out, int words, const uint32_t *plane, bool any) {
    for (int i = threadIdx.x; i < words; i += NT) out[i] = any ? plane[i] : 0u;
}
// 8 pixels -> 8 bfloat16 (0x3F80 = 1.0) = one 16-byte store; the caller guarantees 16-byte alignment and npx % 8 == 0
template <int NT>
__device__ __forceinline__ void tc_store_bf16(uint16_t *out, uint32_t npx, const uint32_t *plane, bool any) {
    uint4 *o4 = (uint4 *)out;
    const uint32_t nvec = npx >> 3;
    for (uint32_t j = threadIdx.x; j < nvec; j += NT) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if (any) {
            uint32_t b = (plane[(8u * j) >> 5] >> ((8u * j) & 31)) & 0xffu;
            if (b) {
                auto two = [](uint32_t q) { return ((q & 1u) ? 0x3F80u : 0u) | ((q & 2u) ? 0x3F800000u : 0u); };
                v = make_uint4(two(b), two(b >> 2), two(b >> 4), two(b >> 6));
            }
        }
        tc_st_cs(o4 + j, v);
    }
}

// classes: grid = N*C*n_bands blocks; each owns rows [y_lo, y_hi) of one class plane
__global__ void __launch_bounds__(TC_RASTER_THREADS) tc_raster_classes_kernel(const TcRasterArgs a) {
    extern __shared__ __align__(16) uint32_t plane[];
    const int band = blockIdx.x % a.n_bands;
    const int pc = blockIdx.x / a.n_bands;
    const int env = pc / a.n_classes, c = pc % a.n_classes;
    if (a.mask && !a.mask[env]) return;
    const int y_lo = band * a.rows_per_band;
    const int y_hi = min(a.H, y_lo + a.rows_per_band);
    const int cnt = a.seg_count[(size_t)env * a.n_classes + c];
    uint8_t *out = a.obs + (((size_t)env * a.n_classes + c) * a.H + y_lo) * a.W;
    const size_t nbytes = (size_t)(y_hi - y_lo) * a.W;
    if (cnt > 0) {
        for (int i = threadIdx.x; i < a.plane_words; i += TC_RASTER_THREADS) plane[i] = 0;
        __syncthreads();
        const int32_t *seg = a.seg + ((size_t)env * a.sum_edges + a.edge_off[c]) * 4;
        const int t = a.thickness[env];
        TcPlane pl = {plane, a.H, a.W, y_lo, y_hi, y_lo};
        TcLanes g = {(int)(threadIdx.x & 31), 32};
        for (int k = threadIdx.x >> 5; k < cnt; k += TC_RASTER_THREADS / 32) {
            int4 s4 = *(const int4 *)(seg + 4 * k);
            tc_polyline2(g, pl, s4.x, s4.y, s4.z, s4.w, t);
        }
        __syncthreads();
    }
    tc_store_plane(out, nbytes, plane, cnt > 0);
}

// rgb, large frames: grid = N*n_bands blocks; C class planes of the band; later classes overwrite earlier ones
// (renderer.py:41-43). Segments come from tc_project_kernel; set-up is split by role over the warps like in the fused kernel.
// (Fallback of tc_render_env_banded_kernel, which sets a frame's segments up once instead of once per band.)
// shared memory: [C class planes + pad word][OR of the class planes + pad word][primitive slots]
__host__ __device__ inline size_t tc_raster_rgb_planes_bytes(int C, int plane_words) { return (((size_t)C * plane_words + 1) * 4 + 15) & ~(size_t)15; }
__host__ __device__ inline size_t tc_raster_rgb_any_bytes(int plane_words) { return (((size_t)plane_words + 1) * 4 + 15) & ~(size_t)15; }
__host__ __device__ inline size_t tc_raster_rgb_smem_bytes(int C, int plane_words) {
    return tc_raster_rgb_planes_bytes(C, plane_words) + tc_raster_rgb_any_bytes(plane_words) + (size_t)TC_SETUP_CHUNK * TC_MAX_PRIMS_PER_SEG * sizeof(TcPrim);
}
__global__ void __launch_bounds__(TC_RASTER_THREADS) tc_raster_rgb_kernel(const TcRasterArgs a) {
    extern __shared__ __align__(16) uint32_t planes[];
    __shared__ int list_src[TC_RASTER_THREADS], list_c[TC_RASTER_THREADS], list_n;
    __shared__ uint32_t color24[TC_MAX_CLASSES];
    __shared__ int cls_cnt[TC_MAX_CLASSES];
    const int C = a.n_classes;
    const int band = blockIdx.x % a.n_bands;
    const int env = blockIdx.x / a.n_bands;
    if (a.mask && !a.mask[env]) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid < TC_MAX_CLASSES) {
        color24[tid] = tc_color24_of(a.colors, tid);
        cls_cnt[tid] = tid < C ? a.seg_count[(size_t)env * C + tid] : 0;
    }
    __syncthreads();
    const int y_lo = band * a.rows_per_band;
    const int y_hi = min(a.H, y_lo + a.rows_per_band);
    uint8_t *out = a.obs + ((size_t)env * a.H + y_lo) * a.W * 3;
    int total = 0;
    for (int c = 0; c < C; c++) total += cls_cnt[c];
    bool drew = false;
    if (total > 0) {
        for (int i = tid; i < C * a.plane_words + 1; i += TC_RASTER_THREADS) planes[i] = 0;
        const int t = a.thickness[env];
        TcLanes g = {lane, 32};
        TcPrim *prims = (TcPrim *)((unsigned char *)planes + tc_raster_rgb_planes_bytes(C, a.plane_words) + tc_raster_rgb_any_bytes(a.plane_words));
        for (int win = 0; win < total; win += TC_RASTER_THREADS) {
            // segments of this window that can touch the band's rows (all primitives stay within t+2 rows of the end points)
            if (tid == 0) list_n = 0;
            __syncthreads();
            if (win + tid < total) {
                int k = win + tid, c = 0;
                while (k >= cls_cnt[c]) { k -= cls_cnt[c]; c++; }
                const int src = a.edge_off[c] + k;
                int4 s4 = *(const int4 *)(a.seg + ((size_t)env * a.sum_edges + src) * 4);
                const long long lo = (long long)min(s4.y, s4.w) - t - 2, hi = (long long)max(s4.y, s4.w) + t + 2;
                if (hi >= y_lo && lo < y_hi) {
                    int slot = atomicAdd(&list_n, 1);
                    list_src[slot] = src;
                    list_c[slot] = c;
                }
            }
            __syncthreads();
            const int nlist = list_n;
            drew = drew || nlist > 0;
            for (int base = 0; base < nlist; base += TC_SETUP_CHUNK) {
                const int nseg = min(TC_SETUP_CHUNK, nlist - base);
                for (int i = tid; i < nseg * TC_MAX_PRIMS_PER_SEG; i += TC_RASTER_THREADS) prims[i].kind = TC_PRIM_NONE;
                __syncthreads();
                if (warp < TC_N_ROLES && lane < nseg) {
                    int4 s4 = *(const int4 *)(a.seg + ((size_t)env * a.sum_edges + list_src[base + lane]) * 4);
                    tc_polyline_setup(a.W, a.H, s4.x, s4.y, s4.z, s4.w, t, warp, prims + lane * TC_MAX_PRIMS_PER_SEG);
                }
                __syncthreads();
                for (int p = warp; p < nseg * TC_MAX_PRIMS_PER_SEG; p += TC_RASTER_THREADS / 32)
                    if (prims[p].kind != TC_PRIM_NONE) {
                        TcPlane pl = {planes + (size_t)list_c[base + p / TC_MAX_PRIMS_PER_SEG] * a.plane_words, a.H, a.W, y_lo, y_hi, y_lo};
                        tc_prim_draw(g, pl, prims[p]);
                    }
                __syncthreads();
            }
        }
    }
    // a frame is mostly background: the OR of the class planes tells the composition which 6-pixel windows have anything in them
    uint32_t *any_plane = (uint32_t *)((unsigned char *)planes + tc_raster_rgb_planes_bytes(C, a.plane_words));
    if (drew) {
        for (int i = tid; i <= a.plane_words; i += TC_RASTER_THREADS) {
            uint32_t v = 0;
            if (i < a.plane_words)
                for (int c = 0; c < C; c++) v |= planes[(size_t)c * a.plane_words + i];
            any_plane[i] = v;
        }
        __syncthreads();
    }
    tc_store_rgb<TC_RASTER_THREADS>(out, (uint32_t)((y_hi - y_lo) * a.W), planes, (uint32_t)a.plane_words * 32u, C, color24, drew, any_plane);
}

#define TC_RGBE_MAX_SEGS 48   // segments whose primitive slots a block-per-env banded kernel keeps in shared memory at once

// ------------------------------------------------------------------------------------------------ fused camera pass + rasterise + store
// classes, single band: a block per (env, class) runs the camera pass in shared memory, keeps the segments on chip,
// rasterises them into the bit plane and streams the plane out. The latency of the geometry of one block hides behind
// the stores of the other blocks resident on the SM; no segment list goes through global memory.
struct TcRenderArgs {
    const TcClassBlob *cblob_desc; // [C] device
    const unsigned char *cblob;    // class blobs (global)
    int n_envs, n_classes, max_nodes, max_edges, max_cblob_bytes;
    int H, W;
    int plane_words;           // words of the full-frame bit plane (incl. pad word)
    const double *pose;        // [N,12]
    const double *cam;         // [N,TC_CAM_N]
    const int32_t *thickness;  // [N]
    const uint8_t *mask;       // optional
    uint8_t *obs;              // [N,C,H,W]
    long long *timeline;       // optional debug [N*C][10]: smid, clock at start / tables landed / geometry done / raster done / end
};

// shared memory: [union{ camera-pass scratch + the class's tables (TMA) | bit plane }][segment list][primitive slots][one byte per
// edge, unused: it keeps the block's footprint, which decides the blocks per SM and (tc_create) which frames take this kernel]
__host__ __device__ inline size_t tc_render_scratch_bytes(int max_nodes) { return (tc_proj_smem_bytes(max_nodes) + 127) & ~(size_t)127; }
__host__ __device__ inline size_t tc_render_union_bytes(int max_nodes, int max_cblob_bytes, int plane_words) {
    size_t a = tc_render_scratch_bytes(max_nodes) + (size_t)max_cblob_bytes, b = (size_t)plane_words * 4;
    return ((a > b ? a : b) + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t tc_render_segs_bytes(int max_edges) { return (size_t)(max_edges > 0 ? max_edges : 1) * 16; }
__host__ __device__ inline size_t tc_render_smem_bytes(int max_nodes, int max_edges, int max_cblob_bytes, int plane_words) {
    return tc_render_union_bytes(max_nodes, max_cblob_bytes, plane_words) + tc_render_segs_bytes(max_edges) +
           (size_t)TC_SETUP_CHUNK * TC_MAX_PRIMS_PER_SEG * sizeof(TcPrim) + (size_t)((max_edges + 15) & ~15);
}

// per-block phase clocks for tools/timeline.py (tc_render_classes_kernel, tc_render_env_kernel): compiled in only with
// -DTC_TIMELINE (the seven 64-bit counters cost registers and spills in the production build). TC_TL runs a statement on
// thread 0 when a timeline is asked for; TC_TL_RECORD writes the block's record [smid, t0, t1, t2, t3, t_end, segments,
// zeroing, set-up, draw] into row blockIdx.x.
#ifdef TC_TIMELINE
#define TC_TL(stmt) do { if (a.timeline && tid == 0) { stmt; } } while (0)
#define TC_TL_DECL long long tl0 = 0, tl1 = 0, tl2 = 0, tl3 = 0, tl_setup = 0, tl_draw = 0, tl_z = 0, tc0 = 0
#define TC_TL_RECORD(t1, cnt) TC_TL(tc_timeline_record(a.timeline, tl0, t1, tl2, tl3, cnt, tl_z, tl_setup, tl_draw))
__device__ __forceinline__ void tc_timeline_record(long long *timeline, long long tl0, long long tl1, long long tl2, long long tl3, int cnt,
                                                   long long tl_z, long long tl_setup, long long tl_draw) {
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    long long *r = timeline + (size_t)blockIdx.x * 10;
    r[0] = smid; r[1] = tl0; r[2] = tl1; r[3] = tl2; r[4] = tl3; r[5] = clock64();
    r[6] = cnt; r[7] = tl_z ? tl_z - tl2 : 0; r[8] = tl_setup; r[9] = tl_draw;
}
#else
#define TC_TL(stmt) do { } while (0)
#define TC_TL_DECL do { } while (0)
#define TC_TL_RECORD(t1, cnt) do { } while (0)
#endif

// NT = 256 threads per block, 4 blocks/SM: the stores dominate
template <int NT, int FMT>
__global__ void __launch_bounds__(NT, 1024 / NT) tc_render_classes_kernel(const TcRenderArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int seg_cnt;
    __shared__ __align__(8) uint64_t bar;
    __shared__ double s_pose[12], s_cam[TC_CAM_N];
    const int env = blockIdx.x / a.n_classes, c = blockIdx.x % a.n_classes;
    if (a.mask && !a.mask[env]) return;
    const int tid = threadIdx.x;
    TC_TL_DECL;
    TC_TL(tl0 = clock64());
    const TcClassBlob cb = a.cblob_desc[c];
    unsigned char *tab_smem = smem_raw + tc_render_scratch_bytes(a.max_nodes);
    if (tid == 0) {
        seg_cnt = 0;
        tc_mbar_init(&bar, 1);
        tc_fence_mbar_init();
        tc_mbar_expect_tx(&bar, (uint32_t)cb.bytes);
        tc_bulk_g2s(tab_smem, a.cblob + cb.offset, (uint32_t)cb.bytes, &bar);
    }
    const int n = cb.n_nodes, m = cb.n_edges;
    int4 *segs = (int4 *)(smem_raw + tc_render_union_bytes(a.max_nodes, a.max_cblob_bytes, a.plane_words));
    uint32_t *plane = (uint32_t *)smem_raw;
    {
        const size_t np = (size_t)((a.max_nodes + 15) & ~15);
        TcProjScratch sc;
        sc.Px = (double *)smem_raw; sc.Py = sc.Px + np; sc.Pz = sc.Py + np;
        sc.ix = (int32_t *)(sc.Pz + np); sc.iy = sc.ix + np;
        uint8_t *fA = (uint8_t *)(sc.iy + np), *fB = fA + np, *rA = fB + np, *rB = rA + np;
        sc.vis = rB + np; sc.front = fA; sc.inr = rA;
        // pose and intrinsics go through shared memory: 17 doubles held in registers by every thread across the whole
        // camera pass would push the kernel over 64 registers, and spills are local-memory traffic behind the stores
        if (tid < 12) s_pose[tid] = a.pose[(size_t)env * 12 + tid];
        else if (tid < 12 + (TC_CAM_MAX_RANGE - TC_CAM_FX + 1)) s_cam[TC_CAM_FX + tid - 12] = a.cam[(size_t)env * TC_CAM_N + TC_CAM_FX + tid - 12];
        __syncthreads();      // barrier init, pose and intrinsics visible to all threads
        const double *pose = s_pose, *cam = s_cam;
        const double max_range = cam[TC_CAM_MAX_RANGE];
        tc_mbar_wait(&bar, 0); // the class's tables have landed in shared memory
        TC_TL(tl1 = clock64());
        const TcClassTables ct = tc_class_tables_from_blob(tab_smem, cb);
        for (int v = tid; v < n; v += NT) {
            double X, Y, Z;
            tc_transform_node(pose, ct.nodes[2 * v], ct.nodes[2 * v + 1], X, Y, Z);
            sc.Px[v] = X; sc.Py[v] = Y; sc.Pz[v] = Z;
            fA[v] = Z < 0;
        }
        __syncthreads();
        for (int v = tid; v < n; v += NT) fB[v] = fA[v] | (uint8_t)tc_clip_pass_node(ct, sc, fA, v, true, -0.0000001);
        __syncthreads();
        for (int v = tid; v < n; v += NT) fA[v] = fB[v] | (uint8_t)tc_clip_pass_node(ct, sc, fB, v, false, -0.0000001);
        __syncthreads();
        for (int v = tid; v < n; v += NT) rA[v] = sc.Pz[v] > -max_range;
        __syncthreads();
        for (int v = tid; v < n; v += NT) rB[v] = rA[v] | (uint8_t)tc_clip_pass_node(ct, sc, rA, v, true, -max_range);
        __syncthreads();
        for (int v = tid; v < n; v += NT) rA[v] = rB[v] | (uint8_t)tc_clip_pass_node(ct, sc, rB, v, false, -max_range);
        __syncthreads();
        for (int v = tid; v < n; v += NT) {
            double u, w;
            tc_project(cam, sc.Px[v], sc.Py[v], sc.Pz[v], u, w);
            sc.ix[v] = tc_np_int32(u);
            sc.iy[v] = tc_np_int32(w);
            sc.vis[v] = (u > 0 && u < a.W && w > 0 && w < a.H && fA[v] && rA[v]) ? 1 : 0;
        }
        __syncthreads();
        // kept edges (camera.py:95); order is irrelevant for a single-colour plane
        for (int e = tid; e < m; e += NT) {
            int n0 = ct.edges[2 * e], n1 = ct.edges[2 * e + 1];
            if (sc.vis[n0] || sc.vis[n1]) {
                int slot = atomicAdd(&seg_cnt, 1);
                segs[slot] = make_int4(sc.ix[n0], sc.iy[n0], sc.ix[n1], sc.iy[n1]);
            }
        }
        __syncthreads(); // scratch and tables are dead from here on; the plane takes their place
    }
    const int cnt = seg_cnt;
    TC_TL(tl2 = clock64());
    if (cnt > 0) {
        for (int i = tid; i < a.plane_words; i += NT) plane[i] = 0;
        __syncthreads();
        TC_TL(tl_z = clock64());
        const int t = a.thickness[env];
        const int warp = tid >> 5, lane = tid & 31;
        TcLanes g = {lane, 32};
        TcPrim *prims = (TcPrim *)((unsigned char *)segs + tc_render_segs_bytes(a.max_edges));
        for (int base = 0; base < cnt; base += TC_SETUP_CHUNK) {
            const int nseg = min(TC_SETUP_CHUNK, cnt - base);
            TC_TL(tc0 = clock64());
            // scalar set-up of up to 16 segments: warp r takes role r (fill spans, one outline edge each, caps) of all of
            // them, lane = segment, so a warp runs one code path
            for (int i = tid; i < nseg * TC_MAX_PRIMS_PER_SEG; i += NT) prims[i].kind = TC_PRIM_NONE;
            __syncthreads();
            if (lane < nseg) {
                int4 s4 = segs[base + lane];
                for (int role = warp; role < TC_N_ROLES; role += NT / 32)
                    tc_polyline_setup(a.W, a.H, s4.x, s4.y, s4.z, s4.w, t, role, prims + lane * TC_MAX_PRIMS_PER_SEG);
            }
            __syncthreads();
            TC_TL(long long x = clock64(); tl_setup += x - tc0; tc0 = x);
            // pixels: the primitives go round-robin to the warps, the pixels / rows of a primitive to the lanes
            for (int p = warp; p < nseg * TC_MAX_PRIMS_PER_SEG; p += (NT / 32))
                if (prims[p].kind != TC_PRIM_NONE) {
                    TcPlane pl = {plane, a.H, a.W, 0, a.H, 0};
                    tc_prim_draw(g, pl, prims[p]);
                }
            __syncthreads();
            TC_TL(tl_draw += clock64() - tc0);
        }
    }
    TC_TL(tl3 = clock64());
    // block (env, class) writes plane blockIdx.x = env * C + class; addressed from blockIdx.x here rather than kept live across
    // the raster phase, which at exactly 64 registers brings spills back
    const size_t hw = (size_t)a.H * a.W;
    if (FMT == TC_FMT_BITS) {
        const int words = (int)((hw + 31) / 32);
        tc_store_bits<NT>((uint32_t *)a.obs + (size_t)blockIdx.x * words, words, plane, cnt > 0);
    } else if (FMT == TC_FMT_BF16)
        tc_store_bf16<NT>((uint16_t *)a.obs + blockIdx.x * hw, (uint32_t)hw, plane, cnt > 0);
    else tc_store_plane<NT>(a.obs + blockIdx.x * hw, hw, plane, cnt > 0);
    TC_TL_RECORD(tl1, cnt);
}

// ------------------------------------------------------------------------------------------------ fused, block per env
// Small frames: a block renders ALL classes of an env into one stacked C*H-row plane (1/C of the barriers, table loads and
// launches of the per-class kernel). A separate kernel from tc_render_classes_kernel because its time goes elsewhere - into
// the camera pass and the rasteriser's set-up, not into the stores - and so that the headline kernel's register allocation
// (64 registers, no spills) is not disturbed. What it does differently:
//  * the camera pass runs on the sub-graph of the ground cell the camera stands in (TcCellBlob, tc_cull.h) instead of the
//    whole map: 3-7x fewer nodes on Knuffingen, and a third of the shared memory (more blocks per SM);
//  * set-up takes 32 segments per round (lane = segment, warp = role) and every primitive is then drawn by ONE thread - the
//    segments of a small frame are a few pixels long, a warp-wide draw keeps 5 lanes busy; a primitive with more than
//    TC_SMALL_PRIM_ITEMS items is handed to the whole warp on the spot;
//  * shared memory is reused aggressively: the segment list overlays the camera-frame coordinates once they are projected,
//    plane and primitive slots overlay the projected coordinates, flags and tables.
#ifndef TC_SMALL_PRIM_ITEMS
#define TC_SMALL_PRIM_ITEMS 24 // measured 12 / 24 / 48 / 96: 24.6 / 24.7 / 23.9 / 23.3 M env-steps/s on Knuffingen 128x160
#endif
#define TC_ENV_CHUNK 32
__device__ __forceinline__ int tc_prim_items(const TcPrim &q) {
    if (q.kind == TC_PRIM_LINE2) return q.a[4] + 1;
    if (q.kind == TC_PRIM_SPAN) return q.a[2] - q.a[1];
    if (q.kind == TC_PRIM_CIRCLE) return 4 * (q.a[2] + 1);
    if (q.kind == TC_PRIM_BRES) return q.a[4] + 1;
    return 0;
}

struct TcRenderEnvArgs {
    const TcCellBlob *cell_desc;   // device
    const unsigned char *cell_blob;
    TcCullGrid grid;
    int n_envs, n_classes;
    int np;                    // node capacity of the scratch arrays (multiple of 16; >= every cell's node count, 24*np >= 17*max edges)
    int max_bytes;             // largest cell blob
    int H, W;
    int plane_words;           // words of the stacked C*H-row bit plane (incl. pad word)
    const double *pose;        // [N,12]
    const double *cam;         // [N,TC_CAM_N]
    const int32_t *thickness;  // [N]
    const uint8_t *mask;       // optional
    uint8_t *obs;
    uint8_t colors[TC_MAX_CLASSES * 3];
    long long *timeline;       // optional debug [N][10], see tools/timeline.py
    int rows_per_band, n_bands, band_words;   // banded variant (large frames): rows per band, bands, words of one class's band plane (incl. pad word)
    int region_bytes;          // packed variant (tc_render_envs_kernel): bytes of one env slot's shared-memory region
    int prim_chunks;           // ... and how many 32-segment chunks its primitive slots hold (1..TC_ENVS_CHUNKS)
};
// shared memory: phase 1 [Px Py Pz | ix iy | 5 flag arrays | cell tables (TMA)]; phase 2 [segments + classes | plane | primitive slots]
__host__ __device__ inline size_t tc_env_np(int max_nodes, int max_edges) {
    size_t need = ((size_t)17 * (max_edges > 0 ? max_edges : 1) + 23) / 24;   // 16 B segment + 1 B class per edge inside 24*np bytes
    size_t np = (size_t)max_nodes > need ? (size_t)max_nodes : need;
    return (np + 15) & ~(size_t)15;
}
__host__ __device__ inline size_t tc_env_off_tables(size_t np) { return (np * 37 + 127) & ~(size_t)127; }
__host__ __device__ inline size_t tc_env_off_plane(size_t np) { return np * 24; }
__host__ __device__ inline size_t tc_env_off_prims(size_t np, int plane_words) { return (np * 24 + (size_t)plane_words * 4 + 15) & ~(size_t)15; }
__host__ __device__ inline size_t tc_env_smem_bytes(size_t np, int max_bytes, int plane_words) {
    size_t a = tc_env_off_tables(np) + (size_t)max_bytes;
    size_t b = tc_env_off_prims(np, plane_words) + (((size_t)TC_ENV_CHUNK * TC_ENV_SEG_WORDS * 4 + 15) & ~(size_t)15);
    return ((a > b ? a : b) + 15) & ~(size_t)15;
}

// The camera pass of the block-per-env kernels (camera.py:52-110) on the sub-graph of the camera's ground cell: transform,
// the four ordered clip passes, projection, visibility (core nodes only), kept edges. In: the cell's tables at tab_smem
// (landing via TMA, mbarrier `bar`), pose and intrinsics in shared memory. Out: *seg_cnt segments as int4 at smem_raw, their
// classes as bytes behind them (segs + d.n_edges); the scratch arrays it used are dead afterwards. All threads call it.
// NT threads (numbered tid = 0..NT-1) work on the env; the block barriers inside are hit by the whole block, so every thread of
// the block must call it (the packed kernel runs one instance per env slot side by side, NT = its threads per env).
// MERGED: the in-range flags of the range passes are taken inside the second near-plane pass instead of in a sweep of their own (one
// barrier and one pass over the nodes less). Only for the kernels that run at 80 registers: in the 64-register kernels it costs 16
// bytes of spills, and a spill there queues behind the observation stores.
template <int NT, bool MERGED = false>
__device__ __forceinline__ void tc_env_camera_pass(unsigned char *smem_raw, size_t np, const unsigned char *tab_smem, const TcCellBlob &d,
                                               uint64_t *bar, const double *pose, const double *cam, int H, int W, int *seg_cnt,
                                               const int tid = threadIdx.x, const uint32_t phase = 0 /* mbarrier parity; 0xffffffff: nothing to wait for */) {
    const int n = d.n_nodes, m = d.n_edges;
    int4 *segs = (int4 *)smem_raw;
    TcProjScratch sc;
    sc.Px = (double *)smem_raw; sc.Py = sc.Px + np; sc.Pz = sc.Py + np;
    sc.ix = (int32_t *)(sc.Pz + np); sc.iy = sc.ix + np;
    uint8_t *fA = (uint8_t *)(sc.iy + np), *fB = fA + np, *rA = fB + np, *rB = rA + np;
    sc.vis = rB + np; sc.front = fA; sc.inr = rA;
    const double max_range = cam[TC_CAM_MAX_RANGE];
    if (phase != 0xffffffffu) tc_mbar_wait(bar, phase); // the cell's tables have landed in shared memory
    const TcClassTables ct = tc_class_tables_from_cell(tab_smem, d);
    const uint8_t *core = tab_smem + d.off_core, *edge_cls = tab_smem + d.off_edge_cls;
    for (int v = tid; v < n; v += NT) {
        double X, Y, Z;
        tc_transform_node(pose, ct.nodes[2 * v], ct.nodes[2 * v + 1], X, Y, Z);
        sc.Px[v] = X; sc.Py[v] = Y; sc.Pz[v] = Z;
        fA[v] = Z < 0;
    }
    __syncthreads();
    // camera.py:70-77 near-plane fix-ups, :80-86 range fix-ups (depths is a live view: evaluated on the moved z): the four
    // ordered passes in ONE loop (one instance of the pass in the code; the flags ping-pong between two arrays)
    for (int pass = 0; pass < 4; pass++) {
        const bool range = pass >= 2, outgoing = (pass & 1) == 0;
        const double tz = range ? -max_range : -0.0000001;
        uint8_t *src = range ? (outgoing ? rA : rB) : (outgoing ? fA : fB), *dst = range ? (outgoing ? rB : rA) : (outgoing ? fB : fA);
        if (!MERGED && pass == 2) {
            for (int v = tid; v < n; v += NT) rA[v] = sc.Pz[v] > -max_range;
            __syncthreads();
        }
        for (int v = tid; v < n; v += NT) {
            dst[v] = src[v] | (uint8_t)tc_clip_pass_node(ct, sc, src, v, outgoing, tz);
            // the in-range flag of the range passes is taken on the z the near-plane passes leave behind (camera.py:80: depths is
            // a live view); a node's z is final for that purpose once its own pass-1 move is done
            if (MERGED && pass == 1) rA[v] = sc.Pz[v] > -max_range;
        }
        __syncthreads();
    }
    for (int v = tid; v < n; v += NT) {
        double u, w;
        tc_project(cam, sc.Px[v], sc.Py[v], sc.Pz[v], u, w);
        sc.ix[v] = tc_np_int32(u);
        sc.iy[v] = tc_np_int32(w);
        sc.vis[v] = (core[v] && u > 0 && u < W && w > 0 && w < H && fA[v] && rA[v]) ? 1 : 0;
    }
    __syncthreads();   // the camera-frame coordinates are dead: the segment list takes their place
    uint8_t *seg_cls = (uint8_t *)(segs + m);
    // kept edges (camera.py:95); order is irrelevant for single-colour planes, and in RGB the classes keep their order
    for (int e = tid; e < m; e += NT) {
        int n0 = ct.edges[2 * e], n1 = ct.edges[2 * e + 1];
        if (sc.vis[n0] || sc.vis[n1]) {
            int slot = atomicAdd(seg_cnt, 1);
            segs[slot] = make_int4(sc.ix[n0], sc.iy[n0], sc.ix[n1], sc.iy[n1]);
            seg_cls[slot] = edge_cls[e];
        }
    }
    __syncthreads();   // projected coordinates, flags and tables are dead: plane and primitive slots take their place
}

// The other phases of the block-per-env kernels, each written once. Where the kernels differ, a template flag or a
// compile-time constant argument selects the difference, so each kernel compiles to what its own copy did.

// Stages view `env` in a block of its own (tc_render_env_kernel, tc_render_env_banded_kernel): thread 0 finds the camera's
// ground cell, whose tables come in with one TMA bulk copy on `bar` (initialised here when init_bar: the banded kernel
// initialises it once for all the views it walks), resets the segment count and publishes the cell's descriptor; warp 1 loads
// the pose and the intrinsics, and in RGB warp 2 the class colours. Ends with a block barrier.
template <bool RGB>
__device__ __forceinline__ void tc_stage_env(const TcRenderEnvArgs &a, int env, unsigned char *tab_smem, uint64_t *bar, bool init_bar, int *seg_cnt,
                                             TcCellBlob *s_desc, double *s_pose, double *s_cam, uint32_t *s_color24) {
    const int tid = threadIdx.x;
    if (tid == 0) {
        // which part of the map can this camera see: its ground cell selects the tables (one TMA bulk copy)
        const TcCellBlob d = a.cell_desc[tc_cull_cell(a.grid, a.pose + (size_t)env * 12)];
        *seg_cnt = 0;
        if (init_bar) {
            tc_mbar_init(bar, 1);
            tc_fence_mbar_init();
        }
        if (d.bytes > 0) {
            tc_mbar_expect_tx(bar, (uint32_t)d.bytes);
            tc_bulk_g2s(tab_smem, a.cell_blob + d.offset, (uint32_t)d.bytes, bar);
        }
        *s_desc = d;
    }
    if (RGB && tid >= 64 && tid < 64 + TC_MAX_CLASSES) s_color24[tid - 64] = tc_color24_of(a.colors, tid - 64);
    if (tid >= 32 && tid < 44) s_pose[tid - 32] = a.pose[(size_t)env * 12 + tid - 32];
    else if (tid >= 44 && tid < 44 + (TC_CAM_MAX_RANGE - TC_CAM_FX + 1)) s_cam[TC_CAM_FX + tid - 44] = a.cam[(size_t)env * TC_CAM_N + TC_CAM_FX + tid - 44];
    __syncthreads();      // barrier init, descriptor, pose and intrinsics visible to all threads
}

// Stages the E view slots of a packed block (tc_render_envs_kernel, tc_prims_kernel; views blockIdx.x * E + e, each with its
// region of a.region_bytes) and runs their camera passes side by side: thread -> (slot j, index of its NT/E threads). A slot past
// the last view or masked out is inactive: the empty cell, thickness 1. `bar` takes one arrival per slot, with its tables' bytes.
template <int NT, int E, bool RGB>
__device__ __forceinline__ void tc_stage_envs(const TcRenderEnvArgs &a, unsigned char *smem_raw, uint64_t *bar, int *seg_cnt, int *s_thick, int *s_active,
                                              TcCellBlob *s_desc, double (*s_pose)[12], double (*s_cam)[TC_CAM_N], uint32_t *s_color24) {
    constexpr int TPE = NT / E;
    if (threadIdx.x == 0) {
        tc_mbar_init(bar, E);
        tc_fence_mbar_init();
    }
    __syncwarp();
    if (threadIdx.x < E) {
        // which part of the map can this env's camera see: its ground cell selects the tables (one TMA bulk copy per env)
        const int e = threadIdx.x, env = blockIdx.x * E + e;
        const bool act = env < a.n_envs && !(a.mask && !a.mask[env]);
        TcCellBlob d;
        if (act) d = a.cell_desc[tc_cull_cell(a.grid, a.pose + (size_t)env * 12)];
        else { d.n_nodes = 0; d.n_edges = 0; d.bytes = 0; d.offset = 0; }
        s_active[e] = act; seg_cnt[e] = 0; s_thick[e] = act ? a.thickness[env] : 1;
        s_desc[e] = d;
        // one arrival per env slot, with its bytes
        if (d.bytes > 0) {
            tc_mbar_expect_tx(bar, (uint32_t)d.bytes);
            tc_bulk_g2s(smem_raw + (size_t)e * a.region_bytes + tc_env_off_tables((size_t)a.np), a.cell_blob + d.offset, (uint32_t)d.bytes, bar);
        } else tc_mbar_arrive(bar);
    }
    if (RGB && threadIdx.x >= 64 && threadIdx.x < 64 + TC_MAX_CLASSES) s_color24[threadIdx.x - 64] = tc_color24_of(a.colors, threadIdx.x - 64);
    if (threadIdx.x >= 32 && threadIdx.x < 32 + E * 17) {
        const int k = threadIdx.x - 32, e = k / 17, i = k % 17, env = blockIdx.x * E + e;
        if (env < a.n_envs) {
            if (i < 12) s_pose[e][i] = a.pose[(size_t)env * 12 + i];
            else s_cam[e][TC_CAM_FX + i - 12] = a.cam[(size_t)env * TC_CAM_N + TC_CAM_FX + i - 12];
        }
    }
    __syncthreads();
    // ---- camera pass (camera.py:52-110) of the E envs side by side
    const int j = threadIdx.x / TPE;
    unsigned char *region = smem_raw + (size_t)j * a.region_bytes;
    tc_env_camera_pass<TPE, true>(region, (size_t)a.np, region + tc_env_off_tables((size_t)a.np), s_desc[j], bar, s_pose[j], s_cam[j], a.H, a.W,
                                  &seg_cnt[j], (int)threadIdx.x - j * TPE);
}

// thread 0: where each slot's segments start in the block's concatenated list, and (s_pref[E]) how many there are
template <int E>
__device__ __forceinline__ void tc_seg_prefix(const int *seg_cnt, int *s_pref) {
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int e = 0; e < E; e++) { s_pref[e] = acc; acc += seg_cnt[e]; }
        s_pref[E] = acc;
    }
}

// marks the primitive slots of a set-up round's nseg segments empty (the set-up fills only the slots a segment needs)
template <int NT>
__device__ __forceinline__ void tc_clear_prim_slots(int32_t *pw, int nseg) {
    for (int i = threadIdx.x; i < nseg * TC_MAX_PRIMS_PER_SEG; i += NT)
        pw[(i / TC_MAX_PRIMS_PER_SEG) * TC_ENV_SEG_WORDS + (i % TC_MAX_PRIMS_PER_SEG) * 8] = TC_PRIM_NONE;
}

// Gathers segments base .. base + nseg - 1 of a packed block's concatenated list for one set-up round: thread i copies segment i
// of the round next to its tag (env slot << 8 | class), and with WITH_GPOS its position in its env's class-sorted list (the
// class's offset s_clsoff plus the segment's rank within its class, rank[e] in slot e's region). Thread 0 resets the task queue.
template <int E, bool WITH_GPOS>
__device__ __forceinline__ void tc_gather_round(const TcRenderEnvArgs &a, const unsigned char *smem_raw, int base, int nseg, const int *s_pref,
                                                const TcCellBlob *s_desc, int4 *s_seg, uint16_t *s_tag, int *s_gpos,
                                                const int (*s_clsoff)[TC_MAX_CLASSES], int *s_task, int *s_nseg, int *s_ntask) {
    if ((int)threadIdx.x < nseg) {   // segment tid of the round: find its env slot, copy it next to its tag
        const int sidx = base + threadIdx.x;
        int e = 0;
#pragma unroll
        for (int k = 1; k < E; k++) e += sidx >= s_pref[k];
        const int i = sidx - s_pref[e];
        const unsigned char *region = smem_raw + (size_t)e * a.region_bytes;
        const int4 *segs = (const int4 *)region;
        const uint8_t cls = ((const uint8_t *)(segs + s_desc[e].n_edges))[i];
        s_seg[threadIdx.x] = segs[i];
        s_tag[threadIdx.x] = (uint16_t)((e << 8) | cls);
        if (WITH_GPOS) s_gpos[threadIdx.x] = s_clsoff[e][cls] + ((const uint16_t *)(region + (size_t)a.np * 24))[i];
    }
    if (threadIdx.x == 0) {
        *s_task = 0; *s_nseg = nseg;
        *s_ntask = ((nseg + TC_ENV_CHUNK - 1) / TC_ENV_CHUNK) * TC_N_ROLES;
    }
}

// Set-up of a packed block's round: (role, chunk) tasks from a queue, lane = segment of the chunk; spans (role 0) are handed out
// first. Each segment's primitives go to its TC_ENV_SEG_WORDS words at pw.
// (Tried in round 2 and rejected: draw tasks in the same queue, each waiting only for the set-up task that fills its slot, so
// that the short roles' primitives are drawn while the spans are still being set up - no barrier between the phases, but
// 9-10 % slower on every small-frame configuration: the ticket order serialises what the barrier let all warps share.)
__device__ __forceinline__ void tc_setup_queue(const TcRenderEnvArgs &a, int *s_task, const int *s_ntask, const int *s_nseg, const int4 *s_seg,
                                               const uint16_t *s_tag, const int *s_thick, int32_t *pw) {
    while (true) {
        int k = 0;
        if ((threadIdx.x & 31) == 0) k = atomicAdd(s_task, 1);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= *s_ntask) break;
        const int nchunks = *s_ntask / TC_N_ROLES;
        const int role = k / nchunks, sl = (k - role * nchunks) * TC_ENV_CHUNK + (threadIdx.x & 31);
        if (sl < *s_nseg) {
            const int4 s4 = s_seg[sl];
            tc_polyline_setup<true>(a.W, a.H, s4.x, s4.y, s4.z, s4.w, s_thick[s_tag[sl] >> 8], role, (TcPrim *)(pw + sl * TC_ENV_SEG_WORDS));
        }
    }
}

// Draws the primitive slots at pw of `nchunks` chunks of 32 segments (nseg of them filled), one thread per primitive: a warp
// takes one slot (= one kind of primitive) of the 32 segments of a chunk. Round 0: every lane draws its own primitive if it is
// short; further rounds: the whole warp draws the long ones (more than TC_SMALL_PRIM_ITEMS items), one after the other - one
// instance of the drawing code serves both. plane_of(sl) is the plane that segment sl of the round draws into.
template <int NT, typename PlaneOf>
__device__ __forceinline__ void tc_draw_prims_by_thread(const int32_t *pw, int nchunks, int nseg, PlaneOf plane_of) {
    const int lane = threadIdx.x & 31;
    for (int p = threadIdx.x; p < nchunks * TC_MAX_PRIMS_PER_SEG * 32; p += NT) {   // uniform trip count within a warp
        const int c = p / (TC_MAX_PRIMS_PER_SEG * 32), slot = (p - c * (TC_MAX_PRIMS_PER_SEG * 32)) >> 5;
        const int sl0 = c * TC_ENV_CHUNK;
        const TcPrim *q = (const TcPrim *)(pw + (sl0 + lane) * TC_ENV_SEG_WORDS + slot * 8);
        int items = 0;
        if (sl0 + lane < nseg && q->kind != TC_PRIM_NONE) items = tc_prim_items(*q);
        unsigned big = __ballot_sync(0xffffffffu, items > TC_SMALL_PRIM_ITEMS);
        bool own = true;
        while (own || big) {
            int src = lane;
            bool active = items > 0 && items <= TC_SMALL_PRIM_ITEMS;
            TcLanes gg = {0, 1};
            if (!own) {
                src = __ffs(big) - 1;
                big &= big - 1;
                active = true;
                gg.lane = lane; gg.n = 32;
            }
            own = false;
            if (active) tc_prim_draw(gg, plane_of(sl0 + src), *(const TcPrim *)(pw + (sl0 + src) * TC_ENV_SEG_WORDS + slot * 8));
        }
    }
}

// Stores view env's stacked C*H-row plane in the output format; any == false: the view has no segments, the frame is zeros.
template <int NT, int FMT>
__device__ __forceinline__ void tc_store_env_frame(const TcRenderEnvArgs &a, int env, const uint32_t *plane, const uint32_t *s_color24, bool any) {
    if (FMT == TC_FMT_RGB)
        tc_store_rgb<NT>(a.obs + (size_t)env * a.H * a.W * 3, (uint32_t)(a.H * a.W), plane, (uint32_t)(a.H * a.W), a.n_classes, s_color24, any);
    else if (FMT == TC_FMT_BITS) {
        // planes are whole words here (the host only selects this format for H*W % 32 == 0)
        const int words = (int)(((size_t)a.H * a.W + 31) / 32) * a.n_classes;
        tc_store_bits<NT>((uint32_t *)a.obs + (size_t)env * words, words, plane, any);
    } else if (FMT == TC_FMT_BF16)
        tc_store_bf16<NT>((uint16_t *)a.obs + (size_t)env * a.n_classes * a.H * a.W, (uint32_t)(a.n_classes * a.H * a.W), plane, any);
    else tc_store_plane_sparse<NT>(a.obs + (size_t)env * a.n_classes * a.H * a.W, (size_t)a.n_classes * a.H * a.W, plane, any);
}

template <int NT, int FMT>
__global__ void __launch_bounds__(NT, 1024 / NT) tc_render_env_kernel(const TcRenderEnvArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int seg_cnt;
    __shared__ __align__(8) uint64_t bar;
    __shared__ double s_pose[12], s_cam[TC_CAM_N];
    __shared__ uint32_t s_color24[TC_MAX_CLASSES];
    __shared__ TcCellBlob s_desc;
    const int env = blockIdx.x;
    if (a.mask && !a.mask[env]) return;
    const int tid = threadIdx.x;
    TC_TL_DECL;
    TC_TL(tl0 = clock64());
    const size_t np = (size_t)a.np;
    unsigned char *tab_smem = smem_raw + tc_env_off_tables(np);
    tc_stage_env<FMT == TC_FMT_RGB>(a, env, tab_smem, &bar, true, &seg_cnt, &s_desc, s_pose, s_cam, s_color24);
    const int n = s_desc.n_nodes, m = s_desc.n_edges;
    int4 *segs = (int4 *)smem_raw;                                   // phase 2 views
    uint32_t *plane = (uint32_t *)(smem_raw + tc_env_off_plane(np));
    int32_t *pw = (int32_t *)(smem_raw + tc_env_off_prims(np, a.plane_words));
    if (n > 0) {
        tc_env_camera_pass<NT>(smem_raw, np, tab_smem, s_desc, &bar, s_pose, s_cam, a.H, a.W, &seg_cnt);
    }
    const int cnt = seg_cnt;
    TC_TL(tl2 = clock64());
    if (cnt > 0) {
        const uint8_t *seg_cls = (const uint8_t *)(segs + m);
        // the plane is zeroed by the warps that have no role in the first set-up round (when the block has more warps than roles)
        constexpr bool ZERO_IN_SETUP = NT / 32 > TC_N_ROLES;
        if (!ZERO_IN_SETUP) {
            for (int i = tid; i < a.plane_words; i += NT) plane[i] = 0;
            __syncthreads();
        }
        TC_TL(tl_z = clock64());
        const int t = a.thickness[env];
        const int warp = tid >> 5, lane = tid & 31;
        for (int base = 0; base < cnt; base += TC_ENV_CHUNK) {
            const int nseg = min(TC_ENV_CHUNK, cnt - base);
            TC_TL(tc0 = clock64());
            tc_clear_prim_slots<NT>(pw, nseg);
            __syncthreads();
            if (ZERO_IN_SETUP && base == 0 && warp >= TC_N_ROLES) {
                for (int i = tid - TC_N_ROLES * 32; i < a.plane_words; i += NT - TC_N_ROLES * 32) plane[i] = 0;
            } else if (lane < nseg) {
                int4 s4 = segs[base + lane];
                for (int role = warp; role < TC_N_ROLES; role += NT / 32)
                    tc_polyline_setup<true>(a.W, a.H, s4.x, s4.y, s4.z, s4.w, t, role, (TcPrim *)(pw + lane * TC_ENV_SEG_WORDS));
            }
            __syncthreads();
            TC_TL(long long x = clock64(); tl_setup += x - tc0; tc0 = x);
            tc_draw_prims_by_thread<NT>(pw, 1, nseg, [&](int sl) {
                const TcPlane pl = {plane, a.H, a.W, 0, a.H, -(int)seg_cls[base + sl] * a.H};
                return pl;
            });
            __syncthreads();
            TC_TL(tl_draw += clock64() - tc0);
        }
    }
    TC_TL(tl3 = clock64());
    tc_store_env_frame<NT, FMT>(a, env, plane, s_color24, cnt > 0);
    TC_TL_RECORD(tl1 ? tl1 : tl0, cnt);   // (the tables' arrival is waited for inside the camera pass: no t1 of its own)
}
#undef TC_TL
#undef TC_TL_DECL
#undef TC_TL_RECORD

// ------------------------------------------------------------------------------------------------ fused, E envs per block
// tc_render_env_kernel leaves most of its lanes idle: a Knuffingen frame has ~120 nodes for 256 threads, ~12 segments for
// the 32 lanes of each set-up warp and ~110 live primitives for 384 draw slots, and the block barriers between the phases cost
// the same whatever the fill. Registers cap the SM at 1024 threads, so the only way to more work in flight is fuller lanes:
// this kernel renders E consecutive envs per block. Their nodes share the threads of the camera pass (NT/E each), their
// segments are concatenated and share the lanes of the set-up and the slots of the draw, and every barrier is paid once per E
// envs. Set-up rounds take TC_ENVS_CHUNKS x 32 segments whose (role, chunk) tasks are handed to the warps from a queue -
// spans first: they are the longest - so that a frame with more than 32 segments does not serialise two set-up rounds.
// Shared memory: E regions laid out like tc_render_env_kernel's (phase 1: scratch + the cell's tables, phase 2: the env's
// segment list and its stacked C*H-row plane), then the primitive slots.
#define TC_ENVS_CHUNKS 2
__host__ __device__ inline size_t tc_envs_region_bytes(size_t np, int max_bytes, int plane_words) {
    size_t a = tc_env_off_tables(np) + (size_t)max_bytes, b = np * 24 + (size_t)plane_words * 4;
    return ((a > b ? a : b) + 127) & ~(size_t)127;
}
__host__ __device__ inline size_t tc_envs_prims_bytes(int chunks) { return (((size_t)chunks * TC_ENV_CHUNK * TC_ENV_SEG_WORDS * 4 + 15) & ~(size_t)15); }
__host__ __device__ inline size_t tc_envs_smem_bytes(int E, size_t np, int max_bytes, int plane_words, int chunks) {
    return (size_t)E * tc_envs_region_bytes(np, max_bytes, plane_words) + tc_envs_prims_bytes(chunks);
}

// 3 blocks per SM: the kernel needs 76-80 registers; capped at 64 (4 blocks) it spills, and a spilled value is a
// local-memory access that queues behind the observation stores of the co-resident blocks (measured: 80 registers at 3 blocks
// per SM beat 64 registers with 72 bytes of spills at 4)
#ifndef TC_ENVS_MIN_BLOCKS
#define TC_ENVS_MIN_BLOCKS(NT) (768 / (NT))
#endif
template <int NT, int FMT, int E>
__global__ void __launch_bounds__(NT, TC_ENVS_MIN_BLOCKS(NT)) tc_render_envs_kernel(const TcRenderEnvArgs a) {
    // Register discipline: the set-up code needs all 64 registers, and a spilled value is a local-memory access that queues
    // behind the observation stores of the co-resident blocks (thousands of cycles each). So nothing is kept in registers across
    // the phases that can be re-read from the kernel parameters (constant bank) or from shared memory.
    constexpr int CAP = TC_ENVS_CHUNKS * TC_ENV_CHUNK; // most segments per set-up round (a.prim_chunks <= TC_ENVS_CHUNKS chunks of 32)
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int seg_cnt[E], s_pref[E + 1], s_thick[E], s_active[E];
    __shared__ __align__(8) uint64_t bar;
    __shared__ double s_pose[E][12], s_cam[E][TC_CAM_N];
    __shared__ uint32_t s_color24[TC_MAX_CLASSES];
    __shared__ TcCellBlob s_desc[E];
    __shared__ int4 s_seg[CAP];        // the round's segments ...
    __shared__ uint16_t s_tag[CAP];    // ... and for each its env slot << 8 | class
    __shared__ int s_task, s_nseg, s_ntask;
#define TC_PLANE(e) ((uint32_t *)(smem_raw + (size_t)(e) * a.region_bytes + (size_t)a.np * 24))
#define TC_PW ((int32_t *)(smem_raw + (size_t)E * a.region_bytes))
    tc_stage_envs<NT, E, FMT == TC_FMT_RGB>(a, smem_raw, &bar, seg_cnt, s_thick, s_active, s_desc, s_pose, s_cam, s_color24);
    tc_seg_prefix<E>(seg_cnt, s_pref);
    // zero the planes of the envs that have segments (the others are stored as zeros without a plane)
    for (int e = 0; e < E; e++)
        if (seg_cnt[e] > 0) {
            uint32_t *pl = TC_PLANE(e);
            for (int i = threadIdx.x; i < a.plane_words; i += NT) pl[i] = 0;
        }
    __syncthreads();
    for (int base = 0; base < s_pref[E]; base += a.prim_chunks * TC_ENV_CHUNK) {
        {
            const int nseg = min(a.prim_chunks * TC_ENV_CHUNK, s_pref[E] - base);
            tc_clear_prim_slots<NT>(TC_PW, nseg);
            tc_gather_round<E, false>(a, smem_raw, base, nseg, s_pref, s_desc, s_seg, s_tag, nullptr, nullptr, &s_task, &s_nseg, &s_ntask);
        }
        __syncthreads();
        tc_setup_queue(a, &s_task, &s_ntask, &s_nseg, s_seg, s_tag, s_thick, TC_PW);
        __syncthreads();
        tc_draw_prims_by_thread<NT>(TC_PW, s_ntask / TC_N_ROLES, s_nseg, [&](int sl) {
            const int tag = s_tag[sl];
            const TcPlane pl = {TC_PLANE(tag >> 8), a.H, a.W, 0, a.H, -(tag & 0xff) * a.H};
            return pl;
        });
        __syncthreads();
    }
    for (int e = 0; e < E; e++)
        if (s_active[e]) tc_store_env_frame<NT, FMT>(a, blockIdx.x * E + e, TC_PLANE(e), s_color24, seg_cnt[e] > 0);
#undef TC_PLANE
#undef TC_PW
}

// ------------------------------------------------------------------------------------------------ large frames, 1 bit per pixel: two kernels
// A 480x640 frame as bit planes is 5 x 38.4 KB: too large for one block to hold all classes, and a block per (env, class) that
// runs the whole pipeline pays the camera pass and the set-up five times per env (the banded kernel above instead pays ten band
// rounds). So the frame is split at the only narrow point of the pipeline, the primitive list (~12 segments x 12 slots x 32 B):
//   tc_prims_kernel       E envs per block like tc_render_envs_kernel - camera pass on the visible-set tables, set-up - but the
//                         primitives go to global memory (L2) instead of being drawn;
//   tc_draw_class_kernel  a block per (env, class): zero a full-frame plane, draw the env's primitives of that class, store the
//                         plane; a class without segments (most `hold` / `area` / `solid` planes) is written as zeros at once.
// Envs with more than TC_PRIMS_CAP segments (long camera ranges) are flagged and rendered by the banded kernel afterwards.
#define TC_PRIMS_CAP 64
#define TC_PRIMS_SEG_WORDS (TC_MAX_PRIMS_PER_SEG * 8)
struct TcPrimsOut {
    int32_t *prims;    // [N][TC_PRIMS_CAP][12][8], an env's segments sorted by class
    int32_t *cls_info; // [N][C]: first segment << 8 | segments of (env, class); -1: the env overflowed. ONE load tells a draw block what to
                       // do - its loads queue behind the observation stores of the co-resident blocks, so every dependent load costs thousands of cycles
    uint8_t *overflow; // [N] 1: the env needs the fallback kernel
};

template <int NT, int E>
__global__ void __launch_bounds__(NT, TC_ENVS_MIN_BLOCKS(NT)) tc_prims_kernel(const TcRenderEnvArgs a, const TcPrimsOut o) {
    constexpr int CAP = TC_ENVS_CHUNKS * TC_ENV_CHUNK;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int seg_cnt[E], s_pref[E + 1], s_thick[E], s_active[E];
    __shared__ __align__(8) uint64_t bar;
    __shared__ double s_pose[E][12], s_cam[E][TC_CAM_N];
    __shared__ TcCellBlob s_desc[E];
    __shared__ int4 s_seg[CAP];
    __shared__ uint16_t s_tag[CAP];   // env slot << 8 | class
    __shared__ int s_gpos[CAP];       // position of the segment in its env's class-sorted list
    __shared__ int s_task, s_nseg, s_ntask;
    __shared__ int s_clscnt[E][TC_MAX_CLASSES], s_clsoff[E][TC_MAX_CLASSES];
#define TC_REGION(e) (smem_raw + (size_t)(e) * a.region_bytes)
#define TC_PW ((int32_t *)(smem_raw + (size_t)E * a.region_bytes))
#define TC_RANK(e) ((uint16_t *)(TC_REGION(e) + (size_t)a.np * 24))   /* rank of a segment within its class: over the dead camera-pass scratch */
    if (threadIdx.x < E * TC_MAX_CLASSES) (&s_clscnt[0][0])[threadIdx.x] = 0;
    tc_stage_envs<NT, E, false>(a, smem_raw, &bar, seg_cnt, s_thick, s_active, s_desc, s_pose, s_cam, nullptr);
    if (threadIdx.x < E) {
        const int e = threadIdx.x, env = blockIdx.x * E + e;
        if (env < a.n_envs) {
            // masked-out envs keep their previous frame: the draw kernel skips them by the same mask, and the fallback kernel by a
            // cleared overflow flag
            const bool ovf = s_active[e] && seg_cnt[e] > TC_PRIMS_CAP;
            o.overflow[env] = ovf ? 1 : 0;
            if (ovf) { seg_cnt[e] = 0; s_active[e] = 2; }   // rendered by the fallback kernel: no set-up here
        }
    }
    __syncthreads();
    // class-sorted order: a segment's rank among the env's segments of its class, then the classes' offsets
    for (int e = 0; e < E; e++) {
        const uint8_t *cls = (const uint8_t *)((const int4 *)TC_REGION(e) + s_desc[e].n_edges);
        for (int i = threadIdx.x; i < seg_cnt[e]; i += NT) TC_RANK(e)[i] = (uint16_t)atomicAdd(&s_clscnt[e][cls[i]], 1);
    }
    tc_seg_prefix<E>(seg_cnt, s_pref);
    __syncthreads();
    if (threadIdx.x < E * a.n_classes) {
        const int e = threadIdx.x / a.n_classes, c = threadIdx.x - e * a.n_classes, env = blockIdx.x * E + e;
        int off = 0;
        for (int k = 0; k < c; k++) off += s_clscnt[e][k];
        s_clsoff[e][c] = off;
        if (env < a.n_envs && s_active[e]) o.cls_info[(size_t)env * a.n_classes + c] = s_active[e] == 2 ? -1 : ((off << 8) | s_clscnt[e][c]);
    }
    __syncthreads();
    for (int base = 0; base < s_pref[E]; base += a.prim_chunks * TC_ENV_CHUNK) {
        {
            const int nseg = min(a.prim_chunks * TC_ENV_CHUNK, s_pref[E] - base);
            tc_clear_prim_slots<NT>(TC_PW, nseg);
            tc_gather_round<E, true>(a, smem_raw, base, nseg, s_pref, s_desc, s_seg, s_tag, s_gpos, s_clsoff, &s_task, &s_nseg, &s_ntask);
        }
        __syncthreads();
        tc_setup_queue(a, &s_task, &s_ntask, &s_nseg, s_seg, s_tag, s_thick, TC_PW);
        __syncthreads();
        // the round's primitives to global memory: consecutive threads write consecutive words of a segment's 12 slots
        for (int i = threadIdx.x; i < s_nseg * TC_PRIMS_SEG_WORDS; i += NT) {
            const int sl = i / TC_PRIMS_SEG_WORDS, wd = i - sl * TC_PRIMS_SEG_WORDS;
            const int env = blockIdx.x * E + (s_tag[sl] >> 8);
            o.prims[((size_t)env * TC_PRIMS_CAP + s_gpos[sl]) * TC_PRIMS_SEG_WORDS + wd] = TC_PW[sl * TC_ENV_SEG_WORDS + wd];
        }
        __syncthreads();
    }
#undef TC_REGION
#undef TC_PW
#undef TC_RANK
}

struct TcDrawArgs {
    int n_envs, n_classes, H, W;
    int plane_words;          // words of one full-frame bit plane (incl. pad word)
    const uint8_t *mask;      // optional
    TcPrimsOut in;
    uint8_t *obs;
};

// FMT: TC_FMT_BITS (u32 [N,C,H*W/32]); the block's plane is the output
template <int NT, int FMT>
__global__ void __launch_bounds__(NT) tc_draw_class_kernel(const TcDrawArgs a) {
    extern __shared__ __align__(128) uint32_t plane[];
    const int env = blockIdx.x / a.n_classes, c = blockIdx.x % a.n_classes;
    const int info = a.in.cls_info[blockIdx.x];   // issued before the mask test: one round trip for both
    if (a.mask && !a.mask[env]) return;
    if (info < 0) return;                  // the env overflowed the primitive buffer: the fallback kernel renders it
    const int tid = threadIdx.x, lane = tid & 31;
    const int n = info & 0xff, first = info >> 8;
    const size_t frame_words = ((size_t)a.H * a.W + 31) / 32;
    uint32_t *out = (uint32_t *)a.obs + ((size_t)env * a.n_classes + c) * frame_words;
    if (n == 0) {   // nothing of this class in view: the plane is zeros
        if ((frame_words & 3) == 0) {
            const uint4 z = make_uint4(0, 0, 0, 0);
            for (size_t i = tid; i < frame_words / 4; i += NT) tc_st_cs((uint4 *)out + i, z);
        } else
            for (size_t i = tid; i < frame_words; i += NT) out[i] = 0u;
        return;
    }
    const TcPlane pl = {plane, a.H, a.W, 0, a.H, 0};
    const TcLanes g = {lane, 32}, g1 = {0, 1};
    const int32_t *base = a.in.prims + (size_t)env * TC_PRIMS_CAP * TC_PRIMS_SEG_WORDS;
    // one thread per primitive slot of the class's segments; long primitives are handed to the whole warp (as in tc_render_env_kernel)
    // (slot p goes to warp p % (NT/32): a class has a few long primitives, and a warp draws its long ones one after the other)
    const int rounds = (n * TC_MAX_PRIMS_PER_SEG + NT - 1) / NT;
    for (int r = 0; r < rounds; r++) {
        const int p = r * NT + lane * (NT / 32) + (tid >> 5);
        TcPrim q;
        q.kind = TC_PRIM_NONE;
        if (p < n * TC_MAX_PRIMS_PER_SEG) {   // both halves at once: the loads are in flight while the plane is zeroed
            const int4 *src = (const int4 *)(base + (size_t)(first + p / TC_MAX_PRIMS_PER_SEG) * TC_PRIMS_SEG_WORDS + (p % TC_MAX_PRIMS_PER_SEG) * 8);
            const int4 lo = src[0], hi = src[1];
            q.kind = lo.x; q.a[0] = lo.y; q.a[1] = lo.z; q.a[2] = lo.w;
            q.a[3] = hi.x; q.a[4] = hi.y; q.a[5] = hi.z; q.a[6] = hi.w;
        }
        if (r == 0) {
            uint4 *p4 = (uint4 *)plane;
            for (int i = tid; i < (a.plane_words + 3) / 4; i += NT) p4[i] = make_uint4(0, 0, 0, 0);
            __syncthreads();
        }
        const int items = q.kind != TC_PRIM_NONE ? tc_prim_items(q) : 0;
        unsigned big = __ballot_sync(0xffffffffu, items > TC_SMALL_PRIM_ITEMS);
        if (items > 0 && items <= TC_SMALL_PRIM_ITEMS) tc_prim_draw(g1, pl, q);
        while (big) {
            const int src = __ffs(big) - 1;
            big &= big - 1;
            TcPrim w;
            w.kind = __shfl_sync(0xffffffffu, q.kind, src);
#pragma unroll
            for (int k = 0; k < 7; k++) w.a[k] = __shfl_sync(0xffffffffu, q.a[k], src);
            tc_prim_draw(g, pl, w);
        }
    }
    __syncthreads();
    if ((frame_words & 3) == 0) {
        for (size_t i = tid; i < frame_words / 4; i += NT) tc_st_cs((uint4 *)out + i, ((const uint4 *)plane)[i]);
    } else
        for (size_t i = tid; i < frame_words; i += NT) out[i] = plane[i];
}

// ------------------------------------------------------------------------------------------------ fused, block per env, banded
// Large frames in the formats whose stores are NOT the bound - RGB (composition work per byte) and 1 bit per pixel (8x fewer
// bytes): a block owns a whole frame. Camera pass on the visible-set sub-graph as in tc_render_env_kernel, set-up of all
// segments once, then the row bands one after the other: zero the C band planes, draw the primitives that can touch the band
// (compact list built by all threads), store. (u8 and bf16 large frames stay with the per-class kernel, which streams at the
// HBM write ceiling.)
// shared memory: phase 1 as tc_render_env_kernel; phase 2 [segments + classes | C band planes + pad | OR plane + pad | primitive slots]
__host__ __device__ inline size_t tc_envb_off_any(size_t np, int C, int band_words) { return np * 24 + tc_raster_rgb_planes_bytes(C, band_words); }
__host__ __device__ inline size_t tc_envb_off_prims(size_t np, int C, int band_words) { return tc_envb_off_any(np, C, band_words) + tc_raster_rgb_any_bytes(band_words); }
__host__ __device__ inline size_t tc_envb_smem_bytes(size_t np, int max_bytes, int C, int band_words) {
    size_t a = tc_env_off_tables(np) + (size_t)max_bytes;
    size_t b = tc_envb_off_prims(np, C, band_words) + (((size_t)TC_RGBE_MAX_SEGS * TC_ENV_SEG_WORDS * 4 + 15) & ~(size_t)15);
    return ((a > b ? a : b) + 15) & ~(size_t)15;
}

#ifndef TC_ENVB_MIN_BLOCKS
#define TC_ENVB_MIN_BLOCKS 4
#endif
template <int FMT>
__global__ void __launch_bounds__(256, TC_ENVB_MIN_BLOCKS) tc_render_env_banded_kernel(const TcRenderEnvArgs a) {
    constexpr int NT = 256;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int seg_cnt;
    __shared__ __align__(8) uint64_t bar;
    __shared__ double s_pose[12], s_cam[TC_CAM_N];
    __shared__ uint32_t s_color24[TC_MAX_CLASSES];
    __shared__ TcCellBlob s_desc;
    __shared__ int seg_lo[TC_RGBE_MAX_SEGS], seg_hi[TC_RGBE_MAX_SEGS];
    __shared__ uint16_t list[TC_RGBE_MAX_SEGS * TC_MAX_PRIMS_PER_SEG];
    __shared__ int list_n;
    __shared__ unsigned band_mask;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int C = a.n_classes;
    const size_t np = (size_t)a.np;
    unsigned char *tab_smem = smem_raw + tc_env_off_tables(np);
    if (tid == 0) {
        tc_mbar_init(&bar, 1);
        tc_fence_mbar_init();
    }
    uint32_t phase = 0;   // parity of the mbarrier's current phase: one TMA copy per rendered env
    // the grid may be smaller than the env count (the fallback launch of the two-kernel path scans a sparse mask with few blocks)
    for (int env = blockIdx.x; env < a.n_envs; env += gridDim.x) {
    if (a.mask && !a.mask[env]) continue;
    __syncthreads();   // the previous env's shared state is dead (and the barrier initialised)
    tc_stage_env<FMT == TC_FMT_RGB>(a, env, tab_smem, &bar, false, &seg_cnt, &s_desc, s_pose, s_cam, s_color24);
    const int n = s_desc.n_nodes, m = s_desc.n_edges;
    int4 *segs = (int4 *)smem_raw;
    uint32_t *planes = (uint32_t *)(smem_raw + np * 24);
    uint32_t *any_plane = (uint32_t *)(smem_raw + tc_envb_off_any(np, C, a.band_words));
    int32_t *pw = (int32_t *)(smem_raw + tc_envb_off_prims(np, C, a.band_words));
    if (n > 0) {
        tc_env_camera_pass<NT>(smem_raw, np, tab_smem, s_desc, &bar, s_pose, s_cam, a.H, a.W, &seg_cnt, threadIdx.x, s_desc.bytes > 0 ? phase : 0xffffffffu);
        if (s_desc.bytes > 0) phase ^= 1u;
    }
    const int total = seg_cnt;
    const uint8_t *seg_cls = (const uint8_t *)(segs + m);
    const int t = a.thickness[env];
    const TcLanes g = {lane, 32};
    // ---- rasteriser: set-up once (or, for more than TC_RGBE_MAX_SEGS segments, per band in rounds), bands in turn
    auto setup = [&](int first, int cnt) {
        if (tid == 0) band_mask = 0;
        tc_clear_prim_slots<NT>(pw, cnt);
        __syncthreads();
        for (int sub = 0; sub < cnt; sub += 32) {
            const int sl = sub + lane;
            if (sl < cnt) {
                const int4 s4 = segs[first + sl];
                if (warp == 7) {   // (the role warps are 0..5) every primitive of a segment stays within t + 2 rows of its end points
                    const long long lo = (long long)min(s4.y, s4.w) - t - 2, hi = (long long)max(s4.y, s4.w) + t + 2;
                    const int ilo = (int)max(lo, (long long)-1), ihi = (int)min(hi, (long long)a.H);
                    seg_lo[sl] = ilo; seg_hi[sl] = ihi;
                    if (ihi >= 0 && ilo < a.H) {
                        const int b0 = max(ilo, 0) / a.rows_per_band, b1 = min(ihi, a.H - 1) / a.rows_per_band;
                        unsigned mk = a.n_bands > 32 ? 0xffffffffu : 0u;
                        for (int b = b0; b <= b1 && a.n_bands <= 32; b++) mk |= 1u << b;
                        atomicOr(&band_mask, mk);
                    }
                }
                for (int role = warp; role < TC_N_ROLES; role += NT / 32)
                    tc_polyline_setup<true>(a.W, a.H, s4.x, s4.y, s4.z, s4.w, t, role, (TcPrim *)(pw + sl * TC_ENV_SEG_WORDS));
            }
        }
        __syncthreads();
    };
    auto draw = [&](int first, int cnt, int y_lo, int y_hi) {
        if (tid == 0) list_n = 0;
        __syncthreads();
        for (int p = tid; p < cnt * TC_MAX_PRIMS_PER_SEG; p += NT) {
            const int sl = p / TC_MAX_PRIMS_PER_SEG;
            if (seg_hi[sl] < y_lo || seg_lo[sl] >= y_hi) continue;
            if (pw[sl * TC_ENV_SEG_WORDS + (p % TC_MAX_PRIMS_PER_SEG) * 8] == TC_PRIM_NONE) continue;
            list[atomicAdd(&list_n, 1)] = (uint16_t)p;
        }
        __syncthreads();
        const int ln = list_n;
        for (int i = warp; i < ln; i += NT / 32) {
            const int p = list[i], sl = p / TC_MAX_PRIMS_PER_SEG;
            const TcPrim &q = *(const TcPrim *)(pw + sl * TC_ENV_SEG_WORDS + (p % TC_MAX_PRIMS_PER_SEG) * 8);
            TcPlane pl = {planes + (size_t)seg_cls[first + sl] * a.band_words, a.H, a.W, y_lo, y_hi, y_lo};
            tc_prim_draw(g, pl, q);
        }
    };
    const bool once = total <= TC_RGBE_MAX_SEGS;
    if (once && total > 0) setup(0, total);
    const size_t frame_words = ((size_t)a.H * a.W + 31) / 32;
    for (int band = 0; band < a.n_bands; band++) {
        const int y_lo = band * a.rows_per_band;
        const int y_hi = min(a.H, y_lo + a.rows_per_band);
        const bool drew = once ? (total > 0 && ((band_mask >> (band & 31)) & 1u)) : total > 0;
        if (drew) {
            for (int i = tid; i < C * a.band_words + 1; i += NT) planes[i] = 0;
            __syncthreads();
            if (once) draw(0, total, y_lo, y_hi);
            else
                for (int first = 0; first < total; first += TC_RGBE_MAX_SEGS) {
                    const int cnt = min(TC_RGBE_MAX_SEGS, total - first);
                    setup(first, cnt);
                    draw(first, cnt, y_lo, y_hi);
                    __syncthreads();
                }
            __syncthreads();
            if (FMT == TC_FMT_RGB) {
                for (int i = tid; i <= a.band_words; i += NT) {
                    uint32_t v = 0;
                    if (i < a.band_words)
                        for (int c = 0; c < C; c++) v |= planes[(size_t)c * a.band_words + i];
                    any_plane[i] = v;
                }
                __syncthreads();
            }
        }
        if (FMT == TC_FMT_RGB)
            tc_store_rgb<NT>(a.obs + ((size_t)env * a.H + y_lo) * a.W * 3, (uint32_t)((y_hi - y_lo) * a.W), planes, (uint32_t)a.band_words * 32u, C,
                             s_color24, drew, any_plane);
        else {
            // 1 bit per pixel: the band planes are the output (the host guarantees rows_per_band * W % 32 == 0)
            const int words = (int)(((size_t)(y_hi - y_lo) * a.W + 31) / 32);
            uint32_t *o = (uint32_t *)a.obs + (size_t)env * C * frame_words + ((size_t)y_lo * a.W) / 32;
            for (int c = 0; c < C; c++)
                for (int i = tid; i < words; i += NT) o[(size_t)c * frame_words + i] = drew ? planes[(size_t)c * a.band_words + i] : 0u;
        }
        __syncthreads();   // the next band reuses the planes
    }
    }
}

// ------------------------------------------------------------------------------------------------ bird's-eye view
// tc_set_bev's contract (include/tinycarlo_b200.h). A block per env: every warp takes 32 segments at a time (lane = segment),
// transforms their endpoints straight from the map tables (a few hundred edges: a brute-force pass, no visible-set tables),
// drops the ones cv2 provably draws nothing for (tc_bev_segment) and draws each survivor with all 32 lanes (tc_polyline2)
// into the stacked P*H-row bit plane in shared memory; then the block stores the planes.
#define TC_BEV_THREADS 256
#define TC_BEV_SMEM_MAX (200 * 1024)   // the stacked plane (tinycarlo_b200/config.py bev_params checks the same bound)
struct TcBevArgs {
    const unsigned char *blob;   // map tables (tc_track_tables)
    TcBlobLayout layout;
    const double *sf;            // [N,TC_SF_N]
    const int32_t *si;           // [N,TC_SI_N]
    TcBevGeom g;
    int n_envs, planes, plane_words, format;   // plane_words: words of the stacked plane incl. the pad word
    const uint8_t *mask;         // optional
    uint8_t *out;
};
__host__ __device__ inline size_t tc_bev_smem_bytes(int plane_words) { return ((size_t)plane_words * 4 + 15) & ~(size_t)15; }

__global__ void __launch_bounds__(TC_BEV_THREADS) tc_bev_kernel(const TcBevArgs a) {
    extern __shared__ __align__(16) uint32_t plane[];
    __shared__ int drew;
    const int env = blockIdx.x, tid = threadIdx.x;
    if (a.mask && !a.mask[env]) return;
    const TcTrackTables tt = tc_track_tables(a.blob, a.layout);
    const double *sf = a.sf + (size_t)env * TC_SF_N;
    const int32_t *si = a.si + (size_t)env * TC_SI_N;
    const double x = sf[TC_SF_X], y = sf[TC_SF_Y], c = cos(sf[TC_SF_ROT]), s = sin(sf[TC_SF_ROT]);
    for (int i = tid; i < a.plane_words; i += TC_BEV_THREADS) plane[i] = 0;
    if (tid == 0) drew = 0;
    __syncthreads();
    const int H = a.g.H, W = a.g.W, n_seg = a.layout.sum_edges + (a.g.route ? 4 : 0);
    const TcLanes g = {(int)(tid & 31), 32};
    for (int base = (tid >> 5) * 32; base < n_seg; base += TC_BEV_THREADS) {   // uniform trip count within a warp
        int32_t p[4] = {0, 0, 0, 0};
        int pl_idx = 0;
        const bool keep = base + g.lane < n_seg && tc_bev_segment(tt, a.g, x, y, c, s, si, base + g.lane, p, pl_idx);
        unsigned todo = __ballot_sync(0xffffffffu, keep);
        if (todo && g.lane == 0) drew = 1;
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const int q = __shfl_sync(0xffffffffu, pl_idx, src);
            const TcPlane pl = {plane, H, W, 0, H, -q * H};
            tc_polyline2(g, pl, __shfl_sync(0xffffffffu, p[0], src), __shfl_sync(0xffffffffu, p[1], src), __shfl_sync(0xffffffffu, p[2], src),
                         __shfl_sync(0xffffffffu, p[3], src), a.g.thickness);
        }
    }
    __syncthreads();
    const size_t npx = (size_t)a.planes * H * W;
    if (a.format == TC_OBS_CLASSES_BITS)   // H*W % 32 == 0 (tc_set_bev): the planes are whole words
        tc_store_bits<TC_BEV_THREADS>((uint32_t *)a.out + (size_t)env * (npx / 32), (int)(npx / 32), plane, drew != 0);
    else tc_store_plane_sparse<TC_BEV_THREADS>(a.out + (size_t)env * npx, npx, plane, drew != 0);
}

// ------------------------------------------------------------------------------------------------ blob noise
// NoiseObservationWrapper (tinycarlo/wrapper/observation.py:14-27) on the device: per class, n_blobs filled circles that
// either erase the class mask or OR in the pixels of a randomly chosen class, applied in the reference's order (classes
// ascending, blobs in sequence, in place: a blob sees what earlier blobs did). The draws (tc_noise_draw) and the disc
// (tc_circle_halfwidths) are tc_core.cuh's, shared with the host test build's mirror ht_noise_blobs.
struct TcNoiseArgs {
    int n_envs, n_cams, n_classes, H, W;
    int n_blobs, max_radius;
    uint32_t seed_lo, seed_hi, step, env_offset;
    const uint8_t *mask; // optional, per env
    uint8_t *obs;        // [N*M,C,H,W] u8
};

// a block per view v = env * M + m
__global__ void __launch_bounds__(256) tc_noise_blobs_kernel(const TcNoiseArgs a) {
    __shared__ int hw[1024]; // half width of the filled midpoint circle per |row offset| (radius < 1024)
    __shared__ int bx, by, brad, bcopy, bsrc;
    const int env = blockIdx.x / a.n_cams, cam = blockIdx.x % a.n_cams, tid = threadIdx.x;
    if (a.mask && !a.mask[env]) return;
    const size_t plane = (size_t)a.H * a.W;
    uint8_t *base = a.obs + (size_t)blockIdx.x * a.n_classes * plane;
    for (int c = 0; c < a.n_classes; c++)
        for (int k = 0; k < a.n_blobs; k++) {
            if (tid == 0) {
                const TcBlobDraw d = tc_noise_draw(a.seed_lo, a.seed_hi, (uint32_t)env + a.env_offset, a.step, c, k, cam, a.n_blobs, a.max_radius,
                                                   a.H, a.W, a.n_classes);
                bx = d.x; by = d.y; brad = d.radius; bcopy = d.copy; bsrc = d.src;
                tc_circle_halfwidths(d.radius, hw);
            }
            __syncthreads();
            const int x = bx, y = by, rad = brad, src = bsrc;
            const bool copy = bcopy != 0;
            uint8_t *dst = base + (size_t)c * plane;
            const uint8_t *sp = base + (size_t)src * plane;
            if (!(copy && src == c)) {
                const int side = 2 * rad + 1;
                for (int i = tid; i < side * side; i += 256) {
                    int ry = i / side - rad, rx = i % side - rad;
                    int h = hw[ry < 0 ? -ry : ry];
                    if (h < 0 || rx < -h || rx > h) continue;
                    int px = x + rx, py = y + ry;
                    if ((unsigned)px >= (unsigned)a.W || (unsigned)py >= (unsigned)a.H) continue;
                    size_t o = (size_t)py * a.W + px;
                    if (copy) dst[o] |= sp[o];
                    else dst[o] = 0;
                }
            }
            __syncthreads();
        }
}

// ------------------------------------------------------------------------------------------------ episode statistics
// The per-rank episode statistics that the ranks all-gather at log cadence (episodes finished, truncations, reward sum, env-steps)
// from a step's reward / terminated / truncated tensors in ONE launch: as torch ops this bookkeeping is eight tiny kernels per
// step, a fifth of the device time of a 4096-env step of small frames.
__global__ void __launch_bounds__(256) tc_episode_stats_kernel(const float *reward, const uint8_t *terminated, const uint8_t *truncated, int n, double *acc4) {
    double ep = 0, tr = 0, rw = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const bool t = truncated[i] != 0;
        ep += (terminated[i] != 0 || t) ? 1.0 : 0.0;
        tr += t ? 1.0 : 0.0;
        rw += (double)reward[i];
    }
    for (int off = 16; off > 0; off >>= 1) {
        ep += __shfl_xor_sync(0xffffffffu, ep, off);
        tr += __shfl_xor_sync(0xffffffffu, tr, off);
        rw += __shfl_xor_sync(0xffffffffu, rw, off);
    }
    __shared__ double s[3][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s[0][warp] = ep; s[1][warp] = tr; s[2][warp] = rw; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double v = 0;
        for (int w = 0; w < 8; w++) v += s[threadIdx.x][w];
        atomicAdd(acc4 + threadIdx.x, v);
    }
    if (blockIdx.x == 0 && threadIdx.x == 3) atomicAdd(acc4 + 3, (double)n);
}

// ------------------------------------------------------------------------------------------------ test hook
// layer.py known-answer queries on class 0 (tests only)
__global__ void tc_debug_layer_kernel(const unsigned char *blob, TcBlobLayout L, int op, double px, double py, double ang, int i0, int i1,
                                      int32_t *out_i, double *out_d) {
    TcTrackTables t = tc_track_tables(blob, L);
    TcLanes g = {(int)(threadIdx.x & 31), 32};
    const double *nodes = t.ll_nodes;
    const int32_t *edges = t.ll_edges;
    int m = t.ll_edge_off[1] - t.ll_edge_off[0];
    int ri = 0;
    double rd = 0;
    if (op == 0) ri = tc_nearest_edge(g, nodes, edges, m, px, py, nullptr, 0, 0);
    else if (op == 1) {
        // orientation of laneline edges is not tabulated; compute it into a small local table via atan2 on the device
        int best = -1;
        double bd = 0;
        for (int e = g.lane; e < m; e += g.n) {
            int a = edges[2 * e], b = edges[2 * e + 1];
            double o = atan2(nodes[2 * b + 1] - nodes[2 * a + 1], nodes[2 * b] - nodes[2 * a]);
            if (!(fabs(tc_clip_angle(o - ang)) <= 30.0 * (TC_PI / 180.0))) continue;
            double d = fabs(tc_dist(px, py, nodes[2 * a], nodes[2 * a + 1]) + tc_dist(px, py, nodes[2 * b], nodes[2 * b + 1]));
            if (best < 0 || d < bd) { best = e; bd = d; }
        }
        tc_group_argmin(g, bd, best);
        ri = best;
    } else if (op == 2)
        ri = tc_within_edge_bounds(px, py, nodes[2 * i0], nodes[2 * i0 + 1], nodes[2 * i1], nodes[2 * i1 + 1]) ? 1 : 0;
    else if (op == 3)
        rd = tc_distance_to_edge(px, py, nodes[2 * i0], nodes[2 * i0 + 1], nodes[2 * i1], nodes[2 * i1 + 1]);
    else if (op == 4)
        rd = tc_clip_angle(ang);
    if (threadIdx.x == 0) {
        out_i[0] = ri;
        out_d[0] = rd;
    }
}
