// tc_api.cu — the C ABI of libtinycarlo_b200.so (see include/tinycarlo_b200.h for what each call replaces).
// Host side: table packing/staging, per-env device buffers, launch configuration. No torch, no CPU compute path.
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "tc_kernels.cuh"
#include "tc_cull.h"
#include "tc_pack.h"

// Kernel attributes are per function, not per handle: several handles with different shared-memory needs coexist
// (TinyCarloGroupedVecEnv), so every kernel is simply allowed the device maximum (227 KB opt-in on sm_100).
template <typename K>
static cudaError_t tc_allow_max_smem(K kernel) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - (int)fa.sharedSizeBytes);
}

static thread_local std::string g_last_error;
static int tc_fail(int code, const std::string &msg) {
    g_last_error = msg;
    return code;
}
#define TC_CUDA(expr)                                                                                                        \
    do {                                                                                                                     \
        cudaError_t _e = (expr);                                                                                             \
        if (_e != cudaSuccess) return tc_fail(TC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));               \
    } while (0)

// One set of visible-set tables on the device (tc_cull.h) with the launch geometry derived from it. A handle keeps the sets it
// has built (by the camera reach they were built for), so that returning to an earlier reach - per-episode camera randomisation
// through the single-env drop-in - neither rebuilds on the host nor allocates nor synchronises.
struct TcCullSet {
    double key = -1.0;                 // the reach asked for
    TcCellBlob *d_desc = nullptr;
    unsigned char *d_blob = nullptr;
    TcCullGrid grid{};
    int np = 0, max_bytes = 0, cells = 0, max_nodes = 0;
    size_t env_smem = 0;     // tc_render_env_kernel (small frames)
    size_t envb_smem = 0;    // tc_render_env_banded_kernel (large frames, RGB / 1 bit per pixel); 0: not available
    size_t envs_smem = 0;
    int pack = 0, chunks = 1;   // pack > 0: tc_render_envs_kernel with that many envs per block
    int blocks = 0;             // resident blocks per SM of the packed kernel as chosen (diagnostics)
    double radius = -1.0, mean_nodes = 0.0;
};

struct TcHandle {
    int device = 0;
    int n_envs = 0, C = 0, H = 0, W = 0, obs_format = 0;
    int n_cams = 1, n_views = 0;   // cameras per env; views v = env * n_cams + m, what the render kernels see as their "envs"
    int sum_nodes = 0, sum_edges = 0, max_nodes = 0;
    int wrapped = 0;
    bool car_set = false, cam_set = false;
    int64_t launches = 0;
    TcBlobLayout layout{};
    std::vector<void *> allocs;
    unsigned char *d_blob = nullptr;
    TcClassTables *d_classes = nullptr;
    TcClassBlob *d_cblob_desc = nullptr;
    unsigned char *d_cblob = nullptr;
    int max_cblob_bytes = 0;
    int32_t *d_edge_off = nullptr;
    double *d_sf = nullptr;
    int32_t *d_si = nullptr;
    double *d_car = nullptr, *d_cam = nullptr, *d_pose = nullptr;   // d_cam, d_pose, d_thick: per view
    int32_t *d_thick = nullptr;
    uint8_t *d_view_mask = nullptr;   // [n_views]: the caller's per-env mask spread over the views (rigs only)
    int32_t *d_seg = nullptr, *d_seg_count = nullptr;
    float *d_act_cc = nullptr; // staging for tc_step_host
    int32_t *d_act_man = nullptr;
    float *d_h_reward = nullptr, *d_h_cte = nullptr, *d_h_heading = nullptr;
    uint8_t *d_h_term = nullptr, *d_h_trunc = nullptr;
    uint8_t colors[TC_MAX_CLASSES * 3] = {0};
    // raster launch geometry
    int rows_per_band_cls = 0, n_bands_cls = 0, plane_words_cls = 0;
    int rows_per_band_rgb = 0, n_bands_rgb = 0, plane_words_rgb = 0;
    size_t track_smem = 0, proj_smem = 0, render_smem = 0;
    int max_edges = 0, plane_words_full = 0;
    int n_sms = 148;
    int track_group = 32;       // lanes per env of tc_track_kernel (32 or 8)
    int track_per_thread = 1;   // tc_track_thread_kernel (one thread per env) instead of tc_track_kernel (a warp per env)
    long long *timeline = nullptr;
    bool fused_ok = false;      // tc_render_classes_kernel's block fits (or fused_all)
    int fused_all = 0;          // small frames: a block per env renders all classes (tc_render_env_kernel / tc_render_envs_kernel)
    // block-per-env kernel: visible-set tables (tc_cull.h), rebuilt when the camera parameters change
    std::vector<int32_t> m_node_off, m_edge_off, m_edges; // host copy of the laneline tables (the builder's input)
    std::vector<double> m_nodes;
    // nearest-laneline index of the tracking kernel (tc_cull.h tc_build_near)
    TcNear near_h;                 // geometry (the tables themselves live on the device)
    int32_t *d_near_off = nullptr;
    uint16_t *d_near_edge = nullptr;
    std::vector<TcCullSet> cull_sets;   // every set built so far (freed by tc_destroy)
    int cull_active = 0;                // cull_sets[cull_active] is the active one (tc_cull_set); tc_create installs the first
    int cull_builds = 0, cull_hits = 0;
    double cull_build_ms_last = 0.0, cull_build_ms_total = 0.0;
    int env_words = 0;
    // two-kernel path of large bit-packed frames (tc_prims_kernel + tc_draw_class_kernel): buffers allocated at first use
    TcPrimsOut prims{};
    int envb_rows = 0, envb_bands = 0, envb_words = 0;
    bool cull_built_once = false;
    uint8_t *ar_done = nullptr; // autoreset flags: caller-owned device buffer
    uint8_t *ar_was_reset = nullptr; // optional: which envs the last step reset (caller-owned)
    uint64_t *rng = nullptr;    // spawn streams: caller-owned device buffers
    const int32_t *spawn_points = nullptr;
    int n_spawn_points = 0;
    int32_t *last_spawn = nullptr;
    TcBevDesc bev{};            // bird's-eye view (tc_set_bev): off while bev_out is NULL
    uint8_t *bev_out = nullptr; // caller-owned
    int bev_planes = 0, bev_plane_words = 0;
    // optional per-kernel CUDA-event timing (tc_profile_begin/end)
    bool profiling = false;
    int prof_cap = 0, prof_used = 0; // step slots
    std::vector<cudaEvent_t> prof_ev; // 4 events per slot: before track, after track, after project, after raster
};

template <typename T>
static int tc_dev_alloc(TcHandle *h, T **p, size_t count) {
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, (count ? count : 1) * sizeof(T));
    if (e != cudaSuccess) return tc_fail(TC_ERR_ALLOC, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    h->allocs.push_back(q);
    *p = (T *)q;
    return TC_OK;
}
#define TC_TRY(expr)             \
    do {                         \
        int _r = (expr);         \
        if (_r != TC_OK) return _r; \
    } while (0)

// rows per band so that rows*W*bytes_per_px is a multiple of 16 (vector stores stay aligned band to band when the
// frame base is) and the bit planes fit the shared-memory budget
static void tc_band_geometry(int H, int W, int planes, size_t smem_budget, int *rows_per_band, int *n_bands, int *plane_words) {
    int rows = H;
    auto words = [&](int r) { return (int)(((size_t)r * W + 31) / 32) + 1; };
    while (rows > 1 && (size_t)words(rows) * 4 * planes > smem_budget) rows = (rows + 1) / 2;
    if (rows < H) {
        int q = 16; // rows multiple of 16 keeps every band start 16-byte aligned for any W
        rows = ((rows + q - 1) / q) * q;
        while (rows > q && (size_t)words(rows) * 4 * planes > smem_budget) rows -= q;
        if (rows > H) rows = H;
    }
    *rows_per_band = rows;
    *n_bands = (H + rows - 1) / rows;
    *plane_words = words(rows);
}

static TcMapDesc tc_host_map(const TcHandle *h) {
    TcMapDesc m{};
    m.n_classes = h->C; m.ll_node_off = h->m_node_off.data(); m.ll_edge_off = h->m_edge_off.data();
    m.ll_nodes = h->m_nodes.data(); m.ll_edges = h->m_edges.data();
    return m;
}
// the active visible-set tables and the launch geometry derived from them
static const TcCullSet &tc_cull_set(const TcHandle *h) { return h->cull_sets[h->cull_active]; }
// makes the visible-set tables for camera reach `radius` (< 0: culling off) the active ones: from the handle's cache, or built
// on the host (tc_cull.h, ~50-150 ms for Knuffingen) and copied to the device. Never frees tables a running kernel may read.
static int tc_install_cull(TcHandle *h, double radius) {
    if (const char *ce = getenv("TC_CULL")) if (atoi(ce) == 0) radius = -1.0;
    for (size_t i = 0; i < h->cull_sets.size(); i++)
        if (h->cull_sets[i].key == radius) {
            h->cull_active = (int)i;
            h->cull_hits++;
            return TC_OK;
        }
    const auto t0 = std::chrono::steady_clock::now();
    TcCull cull;
    TcMapDesc m = tc_host_map(h);
    tc_build_cull(&m, radius, 0.25, 0.05, cull);
    TcCullSet c;
    c.key = radius;
    const size_t np = tc_env_np(cull.max_nodes, cull.max_edges);
    const size_t smem = h->fused_all ? tc_env_smem_bytes(np, cull.max_bytes, h->env_words) : 0;
    if (smem > 200 * 1024) return tc_fail(TC_ERR_INVALID, "visible-set tables exceed the shared-memory budget");
    size_t smem_b = h->fused_all ? 0 : tc_envb_smem_bytes(np, cull.max_bytes, h->C, h->envb_words);
    if (smem_b > 110 * 1024 || (h->envb_rows * h->W) % 32 != 0 || h->envb_bands > 1024) smem_b = 0;   // not worth it / not word aligned: other paths
    TC_CUDA(cudaMalloc((void **)&c.d_desc, cull.desc.size() * sizeof(TcCellBlob)));
    cudaError_t e = cudaMalloc((void **)&c.d_blob, std::max<size_t>(cull.blob.size(), 16));
    if (e != cudaSuccess) { cudaFree(c.d_desc); return tc_fail(TC_ERR_ALLOC, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
    h->cull_sets.push_back(c);   // owned by the handle from here on (tc_destroy frees it)
    TC_CUDA(cudaMemcpy(c.d_desc, cull.desc.data(), cull.desc.size() * sizeof(TcCellBlob), cudaMemcpyHostToDevice));
    if (!cull.blob.empty()) TC_CUDA(cudaMemcpy(c.d_blob, cull.blob.data(), cull.blob.size(), cudaMemcpyHostToDevice));
    {
        // The packed small-frame kernel (tc_render_envs_kernel, 3 blocks of 256 threads per SM): E envs per block and 1 or 2
        // 32-segment chunks of primitive slots, chosen for the most envs in flight per SM without dropping below 3 blocks per SM
        // (fewer blocks hide the latency-bound phases worse than fuller lanes gain); E = 1 never beats tc_render_env_kernel
        // (measured), which stays the fallback. TC_ENV_PACK=0 selects the one-env kernel, so that tests reach it where the packed one would run.
        int pack = 0, chunks = 1, nblocks = 0;
        if (h->fused_all) {
            int best = 0;
            for (int ee : {2, 4})
                for (int cc : {2, 1}) {
                    const size_t sm = tc_envs_smem_bytes(ee, np, cull.max_bytes, h->env_words, cc);
                    if (sm > 200 * 1024) continue;
                    int blocks = 0;   // what the device really keeps resident (registers, static + reserved shared memory, carve-out steps)
                    cudaError_t oe = ee == 2 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, tc_render_envs_kernel<256, TC_FMT_U8, 2>, 256, sm)
                                             : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, tc_render_envs_kernel<256, TC_FMT_U8, 4>, 256, sm);
                    if (oe != cudaSuccess) { cudaGetLastError(); continue; }
                    // (at 2 blocks per SM the packed kernel loses to the one-env kernel at 4: config 5's wide cameras, 0.42 vs 0.35 ms)
                    if (blocks >= 3 && ee * blocks > best) { best = ee * blocks; pack = ee; chunks = cc; nblocks = blocks; }
                }
            if (const char *pe = getenv("TC_ENV_PACK")) if (atoi(pe) == 0) pack = 0;
        }
        c.pack = pack; c.chunks = chunks; c.blocks = nblocks;
        c.envs_smem = pack ? tc_envs_smem_bytes(pack, np, cull.max_bytes, h->env_words, chunks) : 0;
    }
    c.grid = cull.grid; c.np = (int)np; c.max_bytes = cull.max_bytes; c.env_smem = smem; c.envb_smem = smem_b;
    c.radius = cull.radius; c.mean_nodes = cull.mean_nodes; c.cells = (int)cull.desc.size(); c.max_nodes = cull.max_nodes;
    h->cull_sets.back() = c;
    h->cull_active = (int)h->cull_sets.size() - 1;
    h->cull_builds++;
    h->cull_build_ms_last = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    h->cull_build_ms_total += h->cull_build_ms_last;
    return TC_OK;
}

extern "C" {

int tc_abi_version(void) { return TC_ABI_VERSION; }
#ifndef TC_SRC_HASH
#define TC_SRC_HASH "unknown"
#endif
const char *tc_build_info(void) { return TC_SRC_HASH; }
const char *tc_last_error(void) { return g_last_error.c_str(); }

int tc_destroy(TcHandle *h) {
    if (!h) return TC_OK;
    cudaSetDevice(h->device);
    for (void *p : h->allocs) cudaFree(p);
    for (TcCullSet &c : h->cull_sets) { cudaFree(c.d_desc); cudaFree(c.d_blob); }
    for (cudaEvent_t e : h->prof_ev) cudaEventDestroy(e);
    delete h;
    return TC_OK;
}

int tc_create(const TcMapDesc *map, const TcSimDesc *sim, int32_t num_envs, int32_t device, TcHandle **out) {
    return tc_create_rig(map, sim, num_envs, 1, device, out);
}

int tc_create_rig(const TcMapDesc *map, const TcSimDesc *sim, int32_t num_envs, int32_t n_cameras, int32_t device, TcHandle **out) {
    if (!map || !sim || !out) return tc_fail(TC_ERR_INVALID, "tc_create: null argument");
    if (num_envs <= 0) return tc_fail(TC_ERR_INVALID, "tc_create: num_envs must be positive");
    if (n_cameras < 1) return tc_fail(TC_ERR_INVALID, "tc_create_rig: n_cameras must be >= 1");
    const int C = map->n_classes;
    if (C <= 0 || C > TC_MAX_CLASSES) return tc_fail(TC_ERR_INVALID, "tc_create: n_classes out of range (1..16)");
    // the per-class render grids index their blocks (view, class) with an int
    if ((int64_t)num_envs * n_cameras * C > INT32_MAX) return tc_fail(TC_ERR_INVALID, "tc_create_rig: num_envs * n_cameras * n_classes exceeds 2^31 - 1");
    if (sim->height <= 0 || sim->width <= 0) return tc_fail(TC_ERR_INVALID, "tc_create: bad resolution");
    if (sim->obs_format < TC_OBS_CLASSES || sim->obs_format > TC_OBS_CLASSES_BF16) return tc_fail(TC_ERR_INVALID, "tc_create: bad obs_format");
    TcPacked pk;
    {
        std::string err = tc_pack_map(map, pk);
        if (!err.empty()) return tc_fail(TC_ERR_INVALID, "tc_create: " + err);
    }
    const int sumN = map->ll_node_off[C], sumE = map->ll_edge_off[C];
    int ndev = 0;
    TC_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return tc_fail(TC_ERR_INVALID, "tc_create: no such CUDA device");
    TC_CUDA(cudaSetDevice(device));

    TcHandle *h = new TcHandle();
    h->device = device; h->n_envs = num_envs; h->n_cams = n_cameras; h->n_views = num_envs * n_cameras; h->C = C; h->H = sim->height; h->W = sim->width; h->obs_format = sim->obs_format;
    h->sum_nodes = sumN; h->sum_edges = sumE;
    memcpy(h->colors, map->ll_colors, (size_t)3 * C);
    h->m_node_off.assign(map->ll_node_off, map->ll_node_off + C + 1);
    h->m_edge_off.assign(map->ll_edge_off, map->ll_edge_off + C + 1);
    h->m_nodes.assign(map->ll_nodes, map->ll_nodes + 2 * (size_t)sumN);
    h->m_edges.assign(map->ll_edges, map->ll_edges + 2 * (size_t)sumE);
    h->max_nodes = pk.max_nodes;
    h->layout = pk.L;
    const TcBlobLayout &L = h->layout;
    h->track_smem = (size_t)L.total_bytes;
    if (h->track_smem > 200 * 1024) { tc_destroy(h); return tc_fail(TC_ERR_INVALID, "tc_create: map tables exceed the shared-memory staging budget (200 KB)"); }

#define TC_TRYH(expr)                  \
    do {                               \
        int _r = (expr);               \
        if (_r != TC_OK) {             \
            tc_destroy(h);             \
            return _r;                 \
        }                              \
    } while (0)
#define TC_CUDAH(expr)                                                                                      \
    do {                                                                                                    \
        cudaError_t _e = (expr);                                                                            \
        if (_e != cudaSuccess) {                                                                            \
            tc_destroy(h);                                                                                  \
            return tc_fail(TC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));                 \
        }                                                                                                   \
    } while (0)

    TC_TRYH(tc_dev_alloc(h, &h->d_blob, pk.blob.size()));
    TC_CUDAH(cudaMemcpy(h->d_blob, pk.blob.data(), pk.blob.size(), cudaMemcpyHostToDevice));
    // per-class tables for the camera pass: views into the device blob + node adjacency CSR
    int32_t *d_adj = nullptr;
    TC_TRYH(tc_dev_alloc(h, &d_adj, pk.adj.size()));
    TC_CUDAH(cudaMemcpy(d_adj, pk.adj.data(), pk.adj.size() * 4, cudaMemcpyHostToDevice));
    std::vector<TcClassTables> cls;
    tc_class_views(map, pk, h->d_blob, d_adj, cls);
    TC_TRYH(tc_dev_alloc(h, &h->d_classes, (size_t)C));
    TC_CUDAH(cudaMemcpy(h->d_classes, cls.data(), sizeof(TcClassTables) * C, cudaMemcpyHostToDevice));
    TC_TRYH(tc_dev_alloc(h, &h->d_cblob, pk.cblob.size()));
    TC_CUDAH(cudaMemcpy(h->d_cblob, pk.cblob.data(), pk.cblob.size(), cudaMemcpyHostToDevice));
    TC_TRYH(tc_dev_alloc(h, &h->d_cblob_desc, (size_t)C));
    TC_CUDAH(cudaMemcpy(h->d_cblob_desc, pk.cblob_desc.data(), sizeof(TcClassBlob) * C, cudaMemcpyHostToDevice));
    h->max_cblob_bytes = pk.max_cblob_bytes;
    TC_TRYH(tc_dev_alloc(h, &h->d_edge_off, (size_t)C + 1));
    TC_CUDAH(cudaMemcpy(h->d_edge_off, map->ll_edge_off, (size_t)(C + 1) * 4, cudaMemcpyHostToDevice));

    {
        // nearest-laneline index: ~16k ground cells over the laneline bounding box + 1 m (farther out the kernel scans all edges)
        TcNear nr;
        tc_build_near(map, 1.0, 16384, nr);
        if (nr.nx > 0) {
            TC_TRYH(tc_dev_alloc(h, &h->d_near_off, nr.off.size()));
            TC_CUDAH(cudaMemcpy(h->d_near_off, nr.off.data(), nr.off.size() * 4, cudaMemcpyHostToDevice));
            TC_TRYH(tc_dev_alloc(h, &h->d_near_edge, nr.edge.size()));
            TC_CUDAH(cudaMemcpy(h->d_near_edge, nr.edge.data(), nr.edge.size() * 2, cudaMemcpyHostToDevice));
            h->near_h = nr;
            h->near_h.off.clear(); h->near_h.off.shrink_to_fit(); h->near_h.edge.clear(); h->near_h.edge.shrink_to_fit();
        }
    }

    // ---- per-env buffers
    const size_t N = (size_t)num_envs, V = (size_t)h->n_views;
    TC_TRYH(tc_dev_alloc(h, &h->d_sf, N * TC_SF_N));
    TC_TRYH(tc_dev_alloc(h, &h->d_si, N * TC_SI_N));
    TC_TRYH(tc_dev_alloc(h, &h->d_car, N * TC_CP_N));
    TC_TRYH(tc_dev_alloc(h, &h->d_cam, V * TC_CAM_N));
    TC_TRYH(tc_dev_alloc(h, &h->d_pose, V * 12));
    TC_TRYH(tc_dev_alloc(h, &h->d_thick, V));
    if (n_cameras > 1) TC_TRYH(tc_dev_alloc(h, &h->d_view_mask, V));
    TC_TRYH(tc_dev_alloc(h, &h->d_seg, V * (size_t)std::max(sumE, 1) * 4));
    TC_TRYH(tc_dev_alloc(h, &h->d_seg_count, V * C));
    TC_TRYH(tc_dev_alloc(h, &h->d_act_cc, N * 2));
    TC_TRYH(tc_dev_alloc(h, &h->d_act_man, N));
    TC_TRYH(tc_dev_alloc(h, &h->d_h_reward, N));
    TC_TRYH(tc_dev_alloc(h, &h->d_h_cte, N));
    TC_TRYH(tc_dev_alloc(h, &h->d_h_heading, N));
    TC_TRYH(tc_dev_alloc(h, &h->d_h_term, N));
    TC_TRYH(tc_dev_alloc(h, &h->d_h_trunc, N));
    TC_CUDAH(cudaMemset(h->d_sf, 0, N * TC_SF_N * sizeof(double)));
    TC_CUDAH(cudaMemset(h->d_si, 0xff, N * TC_SI_N * sizeof(int32_t)));
    TC_CUDAH(cudaMemset(h->d_seg_count, 0, V * C * sizeof(int32_t)));
    TC_CUDAH(cudaMemset(h->d_pose, 0, V * 12 * sizeof(double)));

    // ---- kernel attributes / launch geometry
    h->proj_smem = tc_proj_smem_bytes(h->max_nodes);
    const size_t plane_budget = 48 * 1024;
    tc_band_geometry(h->H, h->W, 1, plane_budget, &h->rows_per_band_cls, &h->n_bands_cls, &h->plane_words_cls);
    // measured on 480x640: 24/32/40/48/64/96 KB -> 3.02/2.64/2.64/2.49/2.32/4.84 ms per 8192 envs
    tc_band_geometry(h->H, h->W, C, 64 * 1024, &h->rows_per_band_rgb, &h->n_bands_rgb, &h->plane_words_rgb);
    for (int c = 0; c < C; c++) h->max_edges = std::max(h->max_edges, map->ll_edge_off[c + 1] - map->ll_edge_off[c]);
    {
        cudaDeviceProp prop;
        TC_CUDAH(cudaGetDeviceProperties(&prop, device));
        h->n_sms = prop.multiProcessorCount;
    }
    h->plane_words_full = (int)(((size_t)h->H * h->W + 31) / 32) + 1;
    {
        // one block per (env, class) with a full-frame plane, or - when all C planes, the union graph and its scratch fit
        // comfortably (small frames) - one block per env rendering all classes: 1/C of the blocks, barriers and table loads
        const int words_all = (int)(((size_t)C * h->H * h->W + 31) / 32) + 1;
        TcCull whole;
        tc_build_cull(map, -1.0, 0.25, 0.05, whole);
        const size_t smem_all = tc_env_smem_bytes(tc_env_np(whole.max_nodes, whole.max_edges), whole.max_bytes, words_all);
        const size_t smem_one = tc_render_smem_bytes(h->max_nodes, h->max_edges, h->max_cblob_bytes, h->plane_words_full);
        // measured (Knuffingen 240x320, 8192 envs): block per env 0.56 ms against 1.05 ms for the per-class blocks, which pay the
        // camera pass and the set-up once per class; beyond ~75 KB a block (3 per SM) the per-class kernel's finer blocks win again
        // (the camera reach, hence the size of the visible-set tables, is not known yet: the plane is what decides)
        const bool all = smem_all <= 100 * 1024 && (size_t)words_all * 4 <= 50 * 1024;
        h->fused_all = all ? 1 : 0;
        h->render_smem = smem_one;
        h->env_words = words_all;
        // C band planes + their OR in 30 KB; with 24*np and the primitive slots of 48 segments: 4 blocks per SM on Knuffingen
        tc_band_geometry(h->H, h->W, C + 1, 30 * 1024, &h->envb_rows, &h->envb_bands, &h->envb_words);
        h->fused_ok = all || smem_one <= 56 * 1024; // >= 4 blocks per SM; larger frames take the banded two-kernel path
    }
#define TC_PREP_RENDER(K)                 \
    TC_CUDAH(tc_allow_max_smem(K));       \
    TC_CUDAH(cudaFuncSetAttribute(K, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared))
    TC_PREP_RENDER((tc_render_env_banded_kernel<TC_FMT_RGB>));
    TC_PREP_RENDER((tc_render_env_banded_kernel<TC_FMT_BITS>));
    TC_PREP_RENDER((tc_prims_kernel<256, 2>));
    TC_PREP_RENDER((tc_draw_class_kernel<256, TC_FMT_BITS>));
    if (h->fused_ok) {
        TC_PREP_RENDER((tc_render_env_kernel<256, TC_FMT_U8>));
        TC_PREP_RENDER((tc_render_env_kernel<256, TC_FMT_RGB>));
        TC_PREP_RENDER((tc_render_env_kernel<256, TC_FMT_BITS>));
        TC_PREP_RENDER((tc_render_env_kernel<256, TC_FMT_BF16>));
#define TC_PREP_ENVS(F) TC_PREP_RENDER((tc_render_envs_kernel<256, F, 2>)); TC_PREP_RENDER((tc_render_envs_kernel<256, F, 4>))
        TC_PREP_ENVS(TC_FMT_U8); TC_PREP_ENVS(TC_FMT_RGB); TC_PREP_ENVS(TC_FMT_BITS); TC_PREP_ENVS(TC_FMT_BF16);
#undef TC_PREP_ENVS
        TC_PREP_RENDER((tc_render_classes_kernel<256, TC_FMT_U8>));
        TC_PREP_RENDER((tc_render_classes_kernel<256, TC_FMT_BITS>));
        TC_PREP_RENDER((tc_render_classes_kernel<256, TC_FMT_BF16>));
    }
#undef TC_PREP_RENDER
    TC_TRYH(tc_install_cull(h, -1.0));   // the whole graph until the camera parameters are known (after the kernels' attributes: it asks for occupancies)
    TC_CUDAH(cudaFuncSetAttribute(tc_track_kernel<32>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TC_CUDAH(cudaFuncSetAttribute(tc_track_kernel<8>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TC_CUDAH(cudaFuncSetAttribute(tc_raster_classes_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TC_CUDAH(cudaFuncSetAttribute(tc_raster_rgb_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TC_CUDAH(tc_allow_max_smem(tc_track_kernel<32>));
    TC_CUDAH(tc_allow_max_smem(tc_track_kernel<8>));
    TC_CUDAH(tc_allow_max_smem(tc_track_thread_kernel));
    TC_CUDAH(cudaFuncSetAttribute(tc_track_thread_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // a warp per env pays off only when there are too few envs to fill the SMs with one thread each
    // measured: 4096 envs 0.033 (8 lanes per env) vs 0.062 ms (thread), 8192 envs 0.035 vs 0.062, 32768 envs 0.187 (warp) vs 0.044 ms:
    // a thread per env once 8 lanes per env would need more than one wave of warps (3 blocks x 8 warps per SM)
    h->track_per_thread = num_envs / 4 > 3 * 8 * h->n_sms ? 1 : 0;
    // below that: 8 lanes per env once a warp per env would need more than one wave of warps (3 blocks x 8 warps per SM), else a warp per env
    h->track_group = num_envs > 3 * 8 * h->n_sms / 2 ? 8 : 32;
    TC_CUDAH(tc_allow_max_smem(tc_project_kernel));
    TC_CUDAH(tc_allow_max_smem(tc_raster_classes_kernel));
    TC_CUDAH(tc_allow_max_smem(tc_raster_rgb_kernel));
    *out = h;
    return TC_OK;
}

int tc_set_car_params(TcHandle *h, const double *dev_params, void *stream) {
    if (!h || !dev_params) return tc_fail(TC_ERR_INVALID, "tc_set_car_params: null argument");
    TC_CUDA(cudaSetDevice(h->device));
    TC_CUDA(cudaMemcpyAsync(h->d_car, dev_params, (size_t)h->n_envs * TC_CP_N * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    h->car_set = true;
    return TC_OK;
}

// reach of the tables to use for cameras that see `radius` far: the first tables of a handle are tight; later ones go up to the
// next step of a geometric ladder (x1.25), so that a reach that keeps changing (camera randomisation per episode) lands on a few
// cached sets instead of a rebuild per change. Tables built for a larger reach are exact for a smaller one, only less tight.
static double tc_cull_ladder(double radius) {
    const double r0 = 0.05;
    if (!(radius > r0)) return r0;
    return r0 * std::pow(1.25, std::ceil(std::log(radius / r0) / std::log(1.25) - 1e-9));
}

int tc_set_camera_params(TcHandle *h, const double *dev_cam, const int32_t *dev_thickness, void *stream) {
    return tc_set_camera_params_host(h, dev_cam, dev_thickness, nullptr, stream);
}

int tc_set_camera_params_host(TcHandle *h, const double *dev_cam, const int32_t *dev_thickness, const double *host_cam, void *stream) {
    if (!h || !dev_cam || !dev_thickness) return tc_fail(TC_ERR_INVALID, "tc_set_camera_params: null argument");
    TC_CUDA(cudaSetDevice(h->device));
    TC_CUDA(cudaMemcpyAsync(h->d_cam, dev_cam, (size_t)h->n_views * TC_CAM_N * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    TC_CUDA(cudaMemcpyAsync(h->d_thick, dev_thickness, (size_t)h->n_views * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    h->cam_set = true;
    // the visible-set tables depend on how far the cameras see: from the caller's host copy of the rows, or read back (synchronises)
    std::vector<double> rows;
    if (!host_cam) {
        rows.resize((size_t)h->n_views * TC_CAM_N);
        TC_CUDA(cudaMemcpyAsync(rows.data(), h->d_cam, rows.size() * sizeof(double), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        TC_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
        host_cam = rows.data();
    }
    // the largest reach over all views: tables built for a nearer camera would drop lines a farther one sees
    double radius = 0.0;
    for (int i = 0; i < h->n_views && radius >= 0; i++) {
        double r = tc_cull_radius_of(host_cam + (size_t)i * TC_CAM_N, h->H, h->W);
        radius = r < 0 ? -1.0 : std::max(radius, r);
    }
    // keep the active tables while they cover the cameras and are not more than twice too wide
    const double active = tc_cull_set(h).radius;
    const bool keep = radius >= 0 && active >= radius && active <= 2.0 * radius;
    if (radius != active && !keep) {
        const bool first = !h->cull_built_once;
        TC_TRY(tc_install_cull(h, radius < 0 || first ? radius : tc_cull_ladder(radius)));
        h->cull_built_once = true;
    }
    return TC_OK;
}

int tc_set_autoreset(TcHandle *h, uint8_t *dev_done) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_set_autoreset: null handle");
    if (dev_done && !h->rng) return tc_fail(TC_ERR_STATE, "tc_set_autoreset: set the spawn streams first (tc_set_spawn_rng)");
    h->ar_done = dev_done;
    return TC_OK;
}

int tc_set_reset_mask(TcHandle *h, uint8_t *dev_was_reset) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_set_reset_mask: null handle");
    h->ar_was_reset = dev_was_reset;
    return TC_OK;
}

int tc_set_spawn_rng(TcHandle *h, uint64_t *dev_rng_state, const int32_t *dev_spawn_points, int32_t n_spawn_points, int32_t *dev_last_spawn) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_set_spawn_rng: null handle");
    if (n_spawn_points < 0 || (n_spawn_points > 0 && !dev_spawn_points)) return tc_fail(TC_ERR_INVALID, "tc_set_spawn_rng: bad spawn_points");
    h->rng = dev_rng_state; h->spawn_points = dev_spawn_points; h->n_spawn_points = n_spawn_points; h->last_spawn = dev_last_spawn;
    if (!dev_rng_state) h->ar_done = nullptr;
    return TC_OK;
}

int tc_set_wrapped(TcHandle *h, int32_t wrapped) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_set_wrapped: null handle");
    h->wrapped = wrapped ? 1 : 0;
    return TC_OK;
}

enum class TcRenderPath {
    ENVS,      // tc_render_envs_kernel: small frames, E envs per block
    ENV,       // tc_render_env_kernel: small frames, one env per block
    PRIMS,     // tc_prims_kernel + tc_draw_class_kernel (+ the banded kernel for overflowing envs): large bit-packed frames
    BANDED,    // tc_render_env_banded_kernel: large RGB / bit-packed frames, bands walked inside a block per env
    CLASSES,   // tc_render_classes_kernel: a block per (env, class), the frame in one plane
    UNFUSED,   // tc_project_kernel + a raster kernel: segment export, frames too large for the fused kernels
};

// The render kernels a launch runs, from the handle's geometry (tc_create, tc_install_cull), the format and what is asked for.
// timeline: per-block phase clocks are wanted (tools/timeline.py), which the packed kernel does not write.
static TcRenderPath tc_render_path(const TcHandle *h, int obs_format, bool segments, bool timeline) {
    using P = TcRenderPath;
    const bool bits = obs_format == TC_OBS_CLASSES_BITS;
    if (segments) return P::UNFUSED;
    const TcCullSet &cs = tc_cull_set(h);
    if (h->fused_all) return cs.pack > 0 && !timeline ? P::ENVS : P::ENV;
    if (cs.envb_smem > 0 && bits && (h->H * h->W) % 128 == 0 && (size_t)h->plane_words_full * 4 <= 64 * 1024) return P::PRIMS;
    if (cs.envb_smem > 0 && (bits || obs_format == TC_OBS_RGB)) return P::BANDED;
    if (h->fused_ok && obs_format != TC_OBS_RGB) return P::CLASSES;
    return P::UNFUSED;
}

// arguments of the block-per-env kernels; plane_words: words of the stacked plane of the small-frame kernels, 0 for the others
static TcRenderEnvArgs tc_render_env_args(const TcHandle *h, const uint8_t *mask, uint8_t *obs, int plane_words) {
    const TcCullSet &cs = tc_cull_set(h);
    TcRenderEnvArgs ea;
    ea.cell_desc = cs.d_desc; ea.cell_blob = cs.d_blob; ea.grid = cs.grid; ea.n_envs = h->n_views; ea.n_classes = h->C;
    ea.np = cs.np; ea.max_bytes = cs.max_bytes; ea.H = h->H; ea.W = h->W; ea.plane_words = plane_words;
    ea.pose = h->d_pose; ea.cam = h->d_cam; ea.thickness = h->d_thick; ea.mask = mask; ea.obs = obs;
    memcpy(ea.colors, h->colors, sizeof(ea.colors));
    ea.timeline = nullptr;
    ea.rows_per_band = h->envb_rows; ea.n_bands = h->envb_bands; ea.band_words = h->envb_words;
    ea.region_bytes = (int)tc_envs_region_bytes((size_t)cs.np, cs.max_bytes, plane_words);
    ea.prim_chunks = 1;
    return ea;
}

// renders the handle's n_views views; mask (NULL = all) is per view
static int tc_launch_render(TcHandle *h, const uint8_t *mask, uint8_t *obs, int obs_format, int32_t *seg_count_out, int32_t *seg_out,
                            cudaStream_t st, cudaEvent_t after_project = nullptr) {
    using P = TcRenderPath;
    const int N = h->n_views, C = h->C;
    const TcCullSet &cs = tc_cull_set(h);
    long long *timeline = mask ? nullptr : h->timeline;
    const P path = tc_render_path(h, obs_format, seg_count_out || seg_out, timeline != nullptr);
    if (obs_format == TC_OBS_CLASSES_BITS || obs_format == TC_OBS_CLASSES_BF16) {
        if (path == P::UNFUSED) return tc_fail(TC_ERR_INVALID, "bit-packed / bf16 observations need the fused render path (frame too large or debug segments requested)");
        if (obs_format == TC_OBS_CLASSES_BF16 && (h->H * h->W) % 8 != 0) return tc_fail(TC_ERR_INVALID, "bf16 observations need H*W to be a multiple of 8");
        if (obs_format == TC_OBS_CLASSES_BITS && (path == P::ENVS || path == P::ENV) && (h->H * h->W) % 32 != 0) return tc_fail(TC_ERR_INVALID, "bit-packed observations of small frames need H*W to be a multiple of 32");
    }
    const P launch = obs ? path : P::UNFUSED;   // without a frame only the camera pass runs
    if (launch == P::PRIMS && !h->prims.prims) {
        TC_TRY(tc_dev_alloc(h, &h->prims.prims, (size_t)N * TC_PRIMS_CAP * TC_PRIMS_SEG_WORDS));
        TC_TRY(tc_dev_alloc(h, &h->prims.cls_info, (size_t)N * C));
        TC_TRY(tc_dev_alloc(h, &h->prims.overflow, (size_t)N));
        TC_CUDA(cudaMemsetAsync(h->prims.cls_info, 0, (size_t)N * C * 4, st));
        TC_CUDA(cudaMemsetAsync(h->prims.overflow, 0, (size_t)N, st));
    }
    if (launch != P::UNFUSED && after_project) TC_CUDA(cudaEventRecord(after_project, st));
    switch (launch) {
    case P::ENVS: {
        TcRenderEnvArgs ea = tc_render_env_args(h, mask, obs, h->env_words);
        ea.prim_chunks = cs.chunks;
        const int E = cs.pack, grid = (N + E - 1) / E;
        const size_t sm = cs.envs_smem;
#define TC_LAUNCH_ENVS(F)                                                                             \
    do {                                                                                              \
        if (E == 4) tc_render_envs_kernel<256, F, 4><<<grid, 256, sm, st>>>(ea);                      \
        else tc_render_envs_kernel<256, F, 2><<<grid, 256, sm, st>>>(ea);                             \
    } while (0)
        if (obs_format == TC_OBS_RGB) TC_LAUNCH_ENVS(TC_FMT_RGB);
        else if (obs_format == TC_OBS_CLASSES_BITS) TC_LAUNCH_ENVS(TC_FMT_BITS);
        else if (obs_format == TC_OBS_CLASSES_BF16) TC_LAUNCH_ENVS(TC_FMT_BF16);
        else TC_LAUNCH_ENVS(TC_FMT_U8);
#undef TC_LAUNCH_ENVS
        break;
    }
    case P::ENV: {
        TcRenderEnvArgs ea = tc_render_env_args(h, mask, obs, h->env_words);
        ea.timeline = timeline;
        const size_t sm = cs.env_smem;
        if (obs_format == TC_OBS_RGB) tc_render_env_kernel<256, TC_FMT_RGB><<<N, 256, sm, st>>>(ea);
        else if (obs_format == TC_OBS_CLASSES_BITS) tc_render_env_kernel<256, TC_FMT_BITS><<<N, 256, sm, st>>>(ea);
        else if (obs_format == TC_OBS_CLASSES_BF16) tc_render_env_kernel<256, TC_FMT_BF16><<<N, 256, sm, st>>>(ea);
        else tc_render_env_kernel<256, TC_FMT_U8><<<N, 256, sm, st>>>(ea);
        break;
    }
    case P::PRIMS: {
        // large frames, 1 bit per pixel: geometry + set-up once per env (primitives to L2), then a block per (env, class) draws and stores;
        // envs with more segments than the primitive buffer holds are flagged and rendered by the banded kernel
        TcRenderEnvArgs ea = tc_render_env_args(h, mask, nullptr, 0);
        const size_t sm1 = tc_envs_smem_bytes(2, (size_t)cs.np, cs.max_bytes, 0, 1);
        tc_prims_kernel<256, 2><<<(N + 1) / 2, 256, sm1, st>>>(ea, h->prims);
        h->launches++;
        TC_CUDA(cudaGetLastError());
        TcDrawArgs da;
        da.n_envs = N; da.n_classes = C; da.H = h->H; da.W = h->W; da.plane_words = h->plane_words_full; da.mask = mask; da.in = h->prims; da.obs = obs;
        tc_draw_class_kernel<256, TC_FMT_BITS><<<N * C, 256, ((size_t)h->plane_words_full * 4 + 15) & ~(size_t)15, st>>>(da);
        h->launches++;
        TC_CUDA(cudaGetLastError());
        ea.mask = h->prims.overflow; ea.obs = obs;   // (the flag is only set for envs the caller's mask selected)
        tc_render_env_banded_kernel<TC_FMT_BITS><<<std::min(N, 2 * h->n_sms), 256, cs.envb_smem, st>>>(ea);   // few blocks scan the (sparse) flags
        break;
    }
    case P::BANDED: {
        // large frames whose stores are not the bound: a block per env, bands walked inside the block
        const TcRenderEnvArgs ea = tc_render_env_args(h, mask, obs, 0);
        if (obs_format == TC_OBS_RGB) tc_render_env_banded_kernel<TC_FMT_RGB><<<N, 256, cs.envb_smem, st>>>(ea);
        else tc_render_env_banded_kernel<TC_FMT_BITS><<<N, 256, cs.envb_smem, st>>>(ea);
        break;
    }
    case P::CLASSES: {
        TcRenderArgs fa;
        fa.cblob_desc = h->d_cblob_desc; fa.cblob = h->d_cblob; fa.max_cblob_bytes = h->max_cblob_bytes; fa.n_envs = N; fa.n_classes = C;
        fa.max_nodes = h->max_nodes; fa.max_edges = h->max_edges;
        fa.H = h->H; fa.W = h->W; fa.plane_words = h->plane_words_full;
        fa.pose = h->d_pose; fa.cam = h->d_cam; fa.thickness = h->d_thick; fa.mask = mask; fa.obs = obs;
        fa.timeline = timeline;
        const int grid = N * C;
        const size_t sm = h->render_smem;
        if (obs_format == TC_OBS_CLASSES_BITS) tc_render_classes_kernel<256, TC_FMT_BITS><<<grid, 256, sm, st>>>(fa);
        else if (obs_format == TC_OBS_CLASSES_BF16) tc_render_classes_kernel<256, TC_FMT_BF16><<<grid, 256, sm, st>>>(fa);
        else tc_render_classes_kernel<256, TC_FMT_U8><<<grid, 256, sm, st>>>(fa);
        break;
    }
    case P::UNFUSED: {
        TcProjArgs pa;
        pa.classes = h->d_classes; pa.n_envs = N; pa.n_classes = C; pa.sum_edges = h->sum_edges; pa.max_nodes = h->max_nodes;
        pa.H = h->H; pa.W = h->W; pa.edge_off = h->d_edge_off; pa.pose = h->d_pose; pa.cam = h->d_cam; pa.mask = mask;
        pa.seg = seg_out ? seg_out : h->d_seg;
        pa.seg_count = seg_count_out ? seg_count_out : h->d_seg_count;
        tc_project_kernel<<<N * C, TC_PROJ_THREADS, h->proj_smem, st>>>(pa);
        h->launches++;
        TC_CUDA(cudaGetLastError());
        if (after_project) TC_CUDA(cudaEventRecord(after_project, st));
        if (!obs) return TC_OK;
        TcRasterArgs ra;
        ra.n_envs = N; ra.n_classes = C; ra.sum_edges = h->sum_edges; ra.H = h->H; ra.W = h->W;
        ra.edge_off = h->d_edge_off; ra.thickness = h->d_thick; ra.mask = mask; ra.seg = pa.seg; ra.seg_count = pa.seg_count; ra.obs = obs;
        memcpy(ra.colors, h->colors, sizeof(ra.colors));
        if (obs_format == TC_OBS_CLASSES) {
            ra.rows_per_band = h->rows_per_band_cls; ra.n_bands = h->n_bands_cls; ra.plane_words = h->plane_words_cls;
            tc_raster_classes_kernel<<<N * C * ra.n_bands, TC_RASTER_THREADS, (size_t)ra.plane_words * 4, st>>>(ra);
        } else {
            ra.rows_per_band = h->rows_per_band_rgb; ra.n_bands = h->n_bands_rgb; ra.plane_words = h->plane_words_rgb;
            tc_raster_rgb_kernel<<<N * ra.n_bands, TC_RASTER_THREADS, tc_raster_rgb_smem_bytes(C, ra.plane_words), st>>>(ra);
        }
        break;
    }
    }
    h->launches++;
    TC_CUDA(cudaGetLastError());
    return TC_OK;
}

// mask: per env; in reset mode a rig's view mask (tc_view_mask) is written alongside
static int tc_launch_track(TcHandle *h, int mode, const float *cc, const int32_t *man, const uint8_t *mask, const int32_t *spawn,
                           const TcOutputs *outs, cudaStream_t st, const double *cc64 = nullptr) {
    TcTrackArgs ta;
    memset(&ta, 0, sizeof(ta));
    ta.blob = h->d_blob; ta.layout = h->layout; ta.n_envs = h->n_envs; ta.n_cams = h->n_cams; ta.mode = mode; ta.wrapped = h->wrapped;
    ta.view_mask = mode == 1 && mask && h->n_cams > 1 ? h->d_view_mask : nullptr;
    ta.sf = h->d_sf; ta.si = h->d_si; ta.car = h->d_car; ta.cam = h->d_cam; ta.pose = h->d_pose;
    ta.act_cc = cc; ta.act_cc64 = cc64; ta.act_man = man; ta.mask = mask; ta.spawn_nodes = spawn;
    ta.near_x0 = h->near_h.x0; ta.near_y0 = h->near_h.y0; ta.near_inv_cell = h->near_h.inv_cell; ta.near_nx = h->near_h.nx; ta.near_ny = h->near_h.ny;
    ta.near_off = h->d_near_off; ta.near_edge = h->d_near_edge;
    ta.done = h->ar_done; ta.was_reset = h->ar_done ? h->ar_was_reset : nullptr; ta.rng = h->rng; ta.spawn_points = h->spawn_points; ta.n_spawn_points = h->n_spawn_points; ta.last_spawn = h->last_spawn;
    if (outs) ta.out = *outs;
    if (h->track_per_thread) {
        tc_track_thread_kernel<<<(h->n_envs + TC_TRACK1_THREADS - 1) / TC_TRACK1_THREADS, TC_TRACK1_THREADS, h->track_smem, st>>>(ta);
    } else if (h->track_group == 8) {
        const int envs_per_block = TC_TRACK_THREADS / 8;
        tc_track_kernel<8><<<(h->n_envs + envs_per_block - 1) / envs_per_block, TC_TRACK_THREADS, h->track_smem, st>>>(ta);
    } else {
        const int envs_per_block = TC_TRACK_THREADS / 32;
        tc_track_kernel<32><<<(h->n_envs + envs_per_block - 1) / envs_per_block, TC_TRACK_THREADS, h->track_smem, st>>>(ta);
    }
    h->launches++;
    TC_CUDA(cudaGetLastError());
    return TC_OK;
}

// the per-view mask the render kernels read for a per-env mask: the caller's own one camera per env, else the handle's
// view mask, which the reset-mode tracking kernel or tc_pose_kernel writes in the same launch sequence
static const uint8_t *tc_view_mask(const TcHandle *h, const uint8_t *mask) { return mask && h->n_cams > 1 ? h->d_view_mask : mask; }

static int tc_launch_bev(TcHandle *h, const uint8_t *mask, cudaStream_t st) {
    TcBevArgs a;
    a.blob = h->d_blob; a.layout = h->layout; a.sf = h->d_sf; a.si = h->d_si;
    a.g.k = h->bev.pixel_per_meter; a.g.col0 = h->bev.car_col; a.g.row0 = h->bev.car_row;
    a.g.H = h->bev.height; a.g.W = h->bev.width; a.g.thickness = h->bev.line_thickness; a.g.route = h->bev.route;
    a.n_envs = h->n_envs; a.planes = h->bev_planes; a.plane_words = h->bev_plane_words; a.format = h->bev.format;
    a.mask = mask; a.out = h->bev_out;
    tc_bev_kernel<<<h->n_envs, TC_BEV_THREADS, tc_bev_smem_bytes(h->bev_plane_words), st>>>(a);
    h->launches++;
    TC_CUDA(cudaGetLastError());
    return TC_OK;
}

int tc_set_bev(TcHandle *h, const TcBevDesc *desc, uint8_t *dev_bev) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_set_bev: null handle");
    if (!dev_bev) {
        h->bev_out = nullptr;
        return TC_OK;
    }
    if (!desc) return tc_fail(TC_ERR_INVALID, "tc_set_bev: null description");
    const TcBevDesc &d = *desc;
    if (d.height <= 0 || d.width <= 0 || d.height > 4096 || d.width > 4096) return tc_fail(TC_ERR_INVALID, "tc_set_bev: bad resolution");
    if (!(std::isfinite(d.pixel_per_meter) && d.pixel_per_meter > 0)) return tc_fail(TC_ERR_INVALID, "tc_set_bev: pixel_per_meter must be finite and > 0");
    if (!std::isfinite(d.car_col) || !std::isfinite(d.car_row)) return tc_fail(TC_ERR_INVALID, "tc_set_bev: car pixel must be finite");
    if (d.line_thickness < 1 || d.line_thickness > 8) return tc_fail(TC_ERR_INVALID, "tc_set_bev: line_thickness must be in 1..8");
    if (d.route != 0 && d.route != 1) return tc_fail(TC_ERR_INVALID, "tc_set_bev: route must be 0 or 1");
    if (d.format != TC_OBS_CLASSES && d.format != TC_OBS_CLASSES_BITS) return tc_fail(TC_ERR_INVALID, "tc_set_bev: format must be TC_OBS_CLASSES or TC_OBS_CLASSES_BITS");
    if (d.format == TC_OBS_CLASSES_BITS && ((size_t)d.height * d.width) % 32 != 0) return tc_fail(TC_ERR_INVALID, "tc_set_bev: the bit-packed format needs H*W to be a multiple of 32");
    const int planes = h->C + d.route;
    if (planes > TC_MAX_CLASSES) return tc_fail(TC_ERR_INVALID, "tc_set_bev: more than 16 planes");
    const size_t words = ((size_t)planes * d.height * d.width + 31) / 32 + 1;
    if (tc_bev_smem_bytes((int)std::min<size_t>(words, 1 << 28)) > TC_BEV_SMEM_MAX) return tc_fail(TC_ERR_INVALID, "tc_set_bev: the BEV planes do not fit the kernel's shared memory");
    TC_CUDA(cudaSetDevice(h->device));
    TC_CUDA(tc_allow_max_smem(tc_bev_kernel));
    h->bev = d; h->bev_out = dev_bev; h->bev_planes = planes; h->bev_plane_words = (int)words;
    return TC_OK;
}

int tc_render_bev(TcHandle *h, const uint8_t *dev_mask, void *stream) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_render_bev: null handle");
    if (!h->bev_out) return tc_fail(TC_ERR_STATE, "tc_render_bev: no BEV set (tc_set_bev)");
    TC_CUDA(cudaSetDevice(h->device));
    return tc_launch_bev(h, dev_mask, (cudaStream_t)stream);
}

int tc_reset(TcHandle *h, const uint8_t *dev_mask, const int32_t *dev_spawn_nodes, const TcOutputs *outs, void *stream) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_reset: null handle");
    if (!dev_spawn_nodes && !h->rng) return tc_fail(TC_ERR_STATE, "tc_reset: no spawn nodes given and no spawn streams set (tc_set_spawn_rng)");
    if (!h->car_set || !h->cam_set) return tc_fail(TC_ERR_STATE, "tc_reset: car/camera parameters not set");
    TC_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    TC_TRY(tc_launch_track(h, 1, nullptr, nullptr, dev_mask, dev_spawn_nodes, outs, st));
    if (outs && (outs->obs || outs->seg_count || outs->seg_i32))
        TC_TRY(tc_launch_render(h, tc_view_mask(h, dev_mask), outs->obs, h->obs_format, outs->seg_count, outs->seg_i32, st));
    if (h->bev_out) TC_TRY(tc_launch_bev(h, dev_mask, st));
    return TC_OK;
}

static int tc_step_impl(TcHandle *h, const float *dev_car_control, const double *dev_car_control64, const int32_t *dev_maneuver,
                        const TcOutputs *outs, void *stream);

int tc_step(TcHandle *h, const float *dev_car_control, const int32_t *dev_maneuver, const TcOutputs *outs, void *stream) {
    if (!dev_car_control) return tc_fail(TC_ERR_INVALID, "tc_step: null argument");
    return tc_step_impl(h, dev_car_control, nullptr, dev_maneuver, outs, stream);
}

int tc_step_f64(TcHandle *h, const double *dev_car_control, const int32_t *dev_maneuver, const TcOutputs *outs, void *stream) {
    if (!dev_car_control) return tc_fail(TC_ERR_INVALID, "tc_step_f64: null argument");
    return tc_step_impl(h, nullptr, dev_car_control, dev_maneuver, outs, stream);
}

static int tc_step_impl(TcHandle *h, const float *dev_car_control, const double *dev_car_control64, const int32_t *dev_maneuver,
                        const TcOutputs *outs, void *stream) {
    if (!h || !dev_maneuver) return tc_fail(TC_ERR_INVALID, "tc_step: null argument");
    if (!h->car_set || !h->cam_set) return tc_fail(TC_ERR_STATE, "tc_step: car/camera parameters not set");
    TC_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool prof = h->profiling && h->prof_used < h->prof_cap;
    cudaEvent_t *ev = prof ? &h->prof_ev[(size_t)4 * h->prof_used] : nullptr;
    if (prof) TC_CUDA(cudaEventRecord(ev[0], st));
    TC_TRY(tc_launch_track(h, 0, dev_car_control, dev_maneuver, nullptr, nullptr, outs, st, dev_car_control64));
    if (prof) TC_CUDA(cudaEventRecord(ev[1], st));
    if (outs && (outs->obs || outs->seg_count || outs->seg_i32))
        TC_TRY(tc_launch_render(h, nullptr, outs->obs, h->obs_format, outs->seg_count, outs->seg_i32, st, prof ? ev[2] : nullptr));
    else if (prof) TC_CUDA(cudaEventRecord(ev[2], st));
    if (prof) {
        TC_CUDA(cudaEventRecord(ev[3], st));
        h->prof_used++;
    }
    if (h->bev_out) TC_TRY(tc_launch_bev(h, nullptr, st));
    return TC_OK;
}

// recompute the camera poses from the current state (after tc_set_state / camera parameter changes): a thread per view
// v = env * n_cams + m; view_mask (optional) receives mask[env] for the render kernels
__global__ void tc_pose_kernel(int n_views, int n_cams, const double *sf, const double *cam, double *pose, const uint8_t *mask, uint8_t *view_mask) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_views) return;
    const int i = v / n_cams;
    if (view_mask) view_mask[v] = mask[i];
    const double *s = sf + (size_t)i * TC_SF_N;
    tc_camera_pose(cam + (size_t)v * TC_CAM_N + TC_CAM_E, s[TC_SF_X], s[TC_SF_Y], cos(s[TC_SF_ROT]), sin(s[TC_SF_ROT]), pose + (size_t)v * 12);
}

int tc_render(TcHandle *h, const uint8_t *dev_mask, uint8_t *dev_obs, int32_t obs_format, int32_t *dev_seg_count, int32_t *dev_seg_i32,
              void *stream) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_render: null handle");
    if (!h->cam_set) return tc_fail(TC_ERR_STATE, "tc_render: camera parameters not set");
    if (obs_format < TC_OBS_CLASSES || obs_format > TC_OBS_CLASSES_BF16) return tc_fail(TC_ERR_INVALID, "tc_render: bad obs_format");
    TC_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t *view_mask = tc_view_mask(h, dev_mask);
    tc_pose_kernel<<<(h->n_views + 127) / 128, 128, 0, st>>>(h->n_views, h->n_cams, h->d_sf, h->d_cam, h->d_pose, dev_mask,
                                                               view_mask != dev_mask ? h->d_view_mask : nullptr);
    h->launches++;
    TC_CUDA(cudaGetLastError());
    return tc_launch_render(h, view_mask, dev_obs, obs_format, dev_seg_count, dev_seg_i32, st);
}

int tc_get_state(TcHandle *h, double *dev_sf, int32_t *dev_si, void *stream) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_get_state: null handle");
    TC_CUDA(cudaSetDevice(h->device));
    if (dev_sf) TC_CUDA(cudaMemcpyAsync(dev_sf, h->d_sf, (size_t)h->n_envs * TC_SF_N * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    if (dev_si) TC_CUDA(cudaMemcpyAsync(dev_si, h->d_si, (size_t)h->n_envs * TC_SI_N * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return TC_OK;
}

int tc_set_state(TcHandle *h, const double *dev_sf, const int32_t *dev_si, void *stream) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_set_state: null handle");
    TC_CUDA(cudaSetDevice(h->device));
    if (dev_sf) TC_CUDA(cudaMemcpyAsync(h->d_sf, dev_sf, (size_t)h->n_envs * TC_SF_N * sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    if (dev_si) TC_CUDA(cudaMemcpyAsync(h->d_si, dev_si, (size_t)h->n_envs * TC_SI_N * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return TC_OK;
}

int tc_step_host(TcHandle *h, const float *host_car_control, const int32_t *host_maneuver, const TcOutputs *dev_outs, float *host_reward,
                 uint8_t *host_terminated, uint8_t *host_truncated, float *host_cte, float *host_heading_error, void *stream) {
    return tc_step_host_obs(h, host_car_control, host_maneuver, dev_outs, host_reward, host_terminated, host_truncated, host_cte,
                            host_heading_error, nullptr, 0, stream);
}

int tc_step_host_obs(TcHandle *h, const float *host_car_control, const int32_t *host_maneuver, const TcOutputs *dev_outs, float *host_reward,
                     uint8_t *host_terminated, uint8_t *host_truncated, float *host_cte, float *host_heading_error, void *host_obs,
                     size_t obs_bytes, void *stream) {
    if (!h || !host_car_control || !host_maneuver) return tc_fail(TC_ERR_INVALID, "tc_step_host: null argument");
    if (host_obs && !(dev_outs && dev_outs->obs)) return tc_fail(TC_ERR_INVALID, "tc_step_host_obs: host_obs needs dev_outs->obs (the device frame buffer)");
    TC_CUDA(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t N = (size_t)h->n_envs;
    TC_CUDA(cudaMemcpyAsync(h->d_act_cc, host_car_control, N * 2 * sizeof(float), cudaMemcpyHostToDevice, st));
    TC_CUDA(cudaMemcpyAsync(h->d_act_man, host_maneuver, N * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    TcOutputs o;
    if (dev_outs) o = *dev_outs; else memset(&o, 0, sizeof(o));
    if (!o.reward) o.reward = h->d_h_reward;
    if (!o.terminated) o.terminated = h->d_h_term;
    if (!o.truncated) o.truncated = h->d_h_trunc;
    if (!o.cte) o.cte = h->d_h_cte;
    if (!o.heading_error) o.heading_error = h->d_h_heading;
    TC_TRY(tc_step(h, h->d_act_cc, h->d_act_man, &o, stream));
    if (host_reward) TC_CUDA(cudaMemcpyAsync(host_reward, o.reward, N * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (host_terminated) TC_CUDA(cudaMemcpyAsync(host_terminated, o.terminated, N, cudaMemcpyDeviceToHost, st));
    if (host_truncated) TC_CUDA(cudaMemcpyAsync(host_truncated, o.truncated, N, cudaMemcpyDeviceToHost, st));
    if (host_cte) TC_CUDA(cudaMemcpyAsync(host_cte, o.cte, N * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (host_heading_error) TC_CUDA(cudaMemcpyAsync(host_heading_error, o.heading_error, N * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (host_obs && obs_bytes) TC_CUDA(cudaMemcpyAsync(host_obs, o.obs, obs_bytes, cudaMemcpyDeviceToHost, st));   // ONE copy for all envs
    TC_CUDA(cudaStreamSynchronize(st));
    return TC_OK;
}

int tc_debug_set_timeline(TcHandle *h, long long *dev_timeline) {
    if (!h) return tc_fail(TC_ERR_INVALID, "tc_debug_set_timeline: null handle");
    h->timeline = dev_timeline;
    return TC_OK;
}

int tc_debug_cull_info(TcHandle *h, double *out4) {
    if (!h || !out4) return tc_fail(TC_ERR_INVALID, "tc_debug_cull_info: null argument");
    const TcCullSet &cs = tc_cull_set(h);
    out4[0] = (h->fused_all || cs.envb_smem > 0) ? cs.radius : -2.0; out4[1] = cs.cells; out4[2] = cs.mean_nodes; out4[3] = cs.max_nodes;
    return TC_OK;
}

int tc_debug_cull_stats(TcHandle *h, double *out4) {
    if (!h || !out4) return tc_fail(TC_ERR_INVALID, "tc_debug_cull_stats: null argument");
    out4[0] = h->cull_builds; out4[1] = h->cull_hits; out4[2] = h->cull_build_ms_last; out4[3] = h->cull_build_ms_total;
    return TC_OK;
}

int tc_debug_render_info(TcHandle *h, int32_t *out8) {
    if (!h || !out8) return tc_fail(TC_ERR_INVALID, "tc_debug_render_info: null argument");
    const TcCullSet &cs = tc_cull_set(h);
    out8[0] = h->fused_all; out8[1] = h->fused_all ? cs.pack : 0; out8[2] = cs.chunks;
    out8[3] = (int32_t)(h->fused_all ? (cs.pack ? cs.envs_smem : cs.env_smem) : h->render_smem);
    out8[4] = h->track_per_thread + 16 * cs.blocks + 1024 * h->track_group; out8[5] = (int32_t)cs.envb_smem; out8[6] = cs.np; out8[7] = cs.max_bytes;
    return TC_OK;
}

int tc_noise_blobs(TcHandle *h, uint8_t *dev_obs, uint64_t seed, uint32_t step, int32_t n_blobs, int32_t max_radius, int32_t env_index_offset,
                   const uint8_t *dev_mask, void *stream) {
    if (!h || !dev_obs) return tc_fail(TC_ERR_INVALID, "tc_noise_blobs: null argument");
    if (n_blobs < 0 || max_radius < 1 || max_radius > 1023) return tc_fail(TC_ERR_INVALID, "tc_noise_blobs: max_radius must be in 1..1023, n_blobs >= 0");
    TC_CUDA(cudaSetDevice(h->device));
    TcNoiseArgs na;
    na.n_envs = h->n_envs; na.n_cams = h->n_cams; na.n_classes = h->C; na.H = h->H; na.W = h->W; na.n_blobs = n_blobs; na.max_radius = max_radius;
    na.seed_lo = (uint32_t)seed; na.seed_hi = (uint32_t)(seed >> 32); na.step = step; na.env_offset = (uint32_t)env_index_offset;
    na.mask = dev_mask; na.obs = dev_obs;
    tc_noise_blobs_kernel<<<h->n_views, 256, 0, (cudaStream_t)stream>>>(na);
    h->launches++;
    TC_CUDA(cudaGetLastError());
    return TC_OK;
}

int tc_episode_stats(const float *dev_reward, const uint8_t *dev_terminated, const uint8_t *dev_truncated, int32_t n, double *dev_acc4, void *stream) {
    if (!dev_reward || !dev_terminated || !dev_truncated || !dev_acc4 || n < 0) return tc_fail(TC_ERR_INVALID, "tc_episode_stats: bad argument");
    if (n == 0) return TC_OK;
    const int blocks = std::min((n + 255) / 256, 64);   // the sum of rewards is a float64 atomic per block: order-dependent in the last bits only
    tc_episode_stats_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(dev_reward, dev_terminated, dev_truncated, n, dev_acc4);
    TC_CUDA(cudaGetLastError());
    return TC_OK;
}

int64_t tc_launch_count(const TcHandle *h) { return h ? h->launches : 0; }

int tc_profile_begin(TcHandle *h, int32_t max_steps) {
    if (!h || max_steps <= 0) return tc_fail(TC_ERR_INVALID, "tc_profile_begin: bad argument");
    TC_CUDA(cudaSetDevice(h->device));
    while ((int)h->prof_ev.size() < 4 * max_steps) {
        cudaEvent_t e;
        TC_CUDA(cudaEventCreate(&e));
        h->prof_ev.push_back(e);
    }
    h->prof_cap = max_steps;
    h->prof_used = 0;
    h->profiling = true;
    return TC_OK;
}

int tc_profile_end(TcHandle *h, double *host_ms_sum /*[3]: track, project, raster*/, int32_t *host_steps) {
    if (!h || !host_ms_sum || !host_steps) return tc_fail(TC_ERR_INVALID, "tc_profile_end: null argument");
    TC_CUDA(cudaSetDevice(h->device));
    host_ms_sum[0] = host_ms_sum[1] = host_ms_sum[2] = 0;
    for (int i = 0; i < h->prof_used; i++) {
        cudaEvent_t *ev = &h->prof_ev[(size_t)4 * i];
        TC_CUDA(cudaEventSynchronize(ev[3]));
        for (int k = 0; k < 3; k++) {
            float ms = 0;
            TC_CUDA(cudaEventElapsedTime(&ms, ev[k], ev[k + 1]));
            host_ms_sum[k] += ms;
        }
    }
    *host_steps = h->prof_used;
    h->profiling = false;
    h->prof_used = 0;
    return TC_OK;
}

int tc_debug_layer_query(TcHandle *h, int32_t op, double px, double py, double a, int32_t i0, int32_t i1, int32_t *dev_out_i,
                         double *dev_out_d, void *stream) {
    if (!h || !dev_out_i || !dev_out_d) return tc_fail(TC_ERR_INVALID, "tc_debug_layer_query: null argument");
    TC_CUDA(cudaSetDevice(h->device));
    tc_debug_layer_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->d_blob, h->layout, op, px, py, a, i0, i1, dev_out_i, dev_out_d);
    h->launches++;
    TC_CUDA(cudaGetLastError());
    return TC_OK;
}

} // extern "C"
