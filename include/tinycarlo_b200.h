/*
 * tinycarlo_b200.h — C ABI of libtinycarlo_b200.so: the B200-native batched replacement of tinycarlo's
 * per-step hot path.  Plain pointers and sizes only; no torch, no C++ types.
 *
 * What each entry point replaces in the reference (paths relative to the reference checkout):
 *   tc_create              TinyCarloEnv.__init__ staging: Map.__init__ (tinycarlo/map.py:9-37), Layer tables
 *                          (tinycarlo/layer.py:15-19), Car.__init__ (tinycarlo/car.py:10-32)
 *   tc_set_car_params      Car.__init__ parameters (tinycarlo/car.py:12-18), one row per env
 *   tc_set_camera_params   Camera.__init__/update_params (tinycarlo/camera.py:12-27,48-50): E (3x4), K, max_range,
 *                          line_thickness per env; E and K are built on the host (camera.py:145-178)
 *   tc_reset               TinyCarloEnv.reset -> Car.reset -> Map.sample_spawn (env.py:101-113, car.py:34-44,
 *                          map.py:51-69) for the masked envs; spawn nodes given by the caller or drawn on the device
 *   tc_set_spawn_rng       the env's np_random (gymnasium seeding of Env.reset(seed), used by map.py:61): one
 *                          numpy-compatible PCG64 stream per env, advanced by the reset paths on the device
 *   tc_set_autoreset       no counterpart (the reference leaves resets to the caller): gymnasium's next-step autoreset
 *                          inside tc_step
 *   tc_step                TinyCarloEnv.step (env.py:115-147): Car.step + find_local_path (car.py:70-148),
 *                          Camera.capture_frame (camera.py:52-110), Renderer.render_camera_frame_classes/_rgb
 *                          (renderer.py:36-51), Car.get_info (car.py:46-68), default reward/termination (env.py:87-99)
 *   tc_render              Camera.capture_frame alone at the current poses (used after tc_reset / tc_set_state)
 *   tc_get_state/set_state direct access to Car.position/rotation/steering_angle/velocity/local_path/last_maneuver
 *   tc_noise_blobs         NoiseObservationWrapper.observation (tinycarlo/wrapper/observation.py:14-27) with a counter-based RNG
 *   tc_step_host           the same step driven with HOST buffers (pinned or pageable): actions are copied in and the
 *                          scalar results copied out inside the call; used for the end-to-end measurement
 *
 * Conventions: every function returns 0 on success or a negative TcError; tc_last_error() gives the message of the
 * last failure on the calling thread. Pointers named dev_* are CUDA device pointers on the handle's device, host_*
 * are host pointers. All work is enqueued on the given stream (a cudaStream_t passed as void*, NULL = legacy
 * default stream) and nothing synchronises unless documented. A handle is not thread-safe; distinct handles are.
 * There is no CPU implementation behind this ABI: without a CUDA device every call fails with TC_ERR_CUDA.
 */
#ifndef TINYCARLO_B200_H
#define TINYCARLO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TC_ABI_VERSION 1
#if defined(__GNUC__)
#define TC_API __attribute__((visibility("default")))
#else
#define TC_API
#endif

typedef struct TcHandle TcHandle;

typedef enum {
    TC_OK = 0,
    TC_ERR_INVALID = -1, /* bad argument */
    TC_ERR_CUDA = -2,    /* CUDA runtime error (message has the cudaError string) */
    TC_ERR_ALLOC = -3,
    TC_ERR_STATE = -4 /* call order (e.g. step before params were set) */
} TcError;

/* Row layouts of the per-env arrays (all row-major, one row per env). */
enum { TC_SF_X = 0, TC_SF_Y, TC_SF_ROT, TC_SF_STEER_DEG, TC_SF_VEL, TC_SF_FRONT_X, TC_SF_FRONT_Y, TC_SF_PAD, TC_SF_N = 8 };
enum { TC_SI_PATH_LEN = 0, TC_SI_LAST_MANEUVER = 1, TC_SI_PATH_NODES = 2 /* 4 x (n0,n1) */, TC_SI_PATH_EDGES = 10 /* 4 */, TC_SI_N = 16 };
enum { TC_CP_WHEELBASE = 0, TC_CP_TRACK_WIDTH, TC_CP_MAX_VELOCITY, TC_CP_MAX_STEERING_DEG, TC_CP_STEERING_SPEED /* NaN = None */,
       TC_CP_MAX_ACCELERATION /* NaN = None */, TC_CP_MAX_DECELERATION, TC_CP_DT, TC_CP_N = 8 };
/* spawn stream row (uint64): PCG64 state hi, lo, increment hi, lo, buffered 32-bit half (bit 32 = valid) */
enum { TC_RNG_HI = 0, TC_RNG_LO, TC_RNG_INC_HI, TC_RNG_INC_LO, TC_RNG_BUF, TC_RNG_N = 5 };
enum { TC_CAM_E = 0 /* 12: row-major 3x4 */, TC_CAM_FX = 12, TC_CAM_FY, TC_CAM_CX, TC_CAM_CY, TC_CAM_MAX_RANGE, TC_CAM_N = 20 };
enum { TC_OBS_CLASSES = 0 /* u8 [N,C,H,W], 0/255 */, TC_OBS_RGB = 1 /* u8 [N,H,W,3], layer colours */,
       /* beyond the reference (SURVEY 8f-1), same masks in the format a policy consumes: */
       TC_OBS_CLASSES_BITS = 2 /* u32 [N,C,ceil(H*W/32)]: bit (y*W+x)%32 of word (y*W+x)/32 = pixel (x,y) */,
       TC_OBS_CLASSES_BF16 = 3 /* bfloat16 [N,C,H,W], 0.0 / 1.0 */ };
/* info_f64 row: cte, heading_error, velocity, reward, then C laneline distances */
enum { TC_INFO_CTE = 0, TC_INFO_HEADING, TC_INFO_VELOCITY, TC_INFO_REWARD, TC_INFO_DIST0 = 4 };

/* Map tables (HOST pointers; copied to the device by tc_create). Class order = key order of "lanelines" in the map JSON. */
typedef struct {
    int32_t n_classes;
    const int32_t *ll_node_off; /* [C+1] first node of each class in ll_nodes */
    const int32_t *ll_edge_off; /* [C+1] first edge of each class in ll_edges */
    const double *ll_nodes;     /* [sumN][2] metres */
    const int32_t *ll_edges;    /* [sumE][2] class-local node ids, JSON order */
    const uint8_t *ll_colors;   /* [C][3] layer_color as stored in the JSON */
    int32_t lp_n_nodes, lp_n_edges;
    const double *lp_nodes;      /* [P][2] metres */
    const int32_t *lp_edges;     /* [Q][2] */
    const double *lp_orient;     /* [Q] atan2(n1-n0) of every lanepath edge, computed by the host libm */
    const double *lp_orient_rev; /* [Q] atan2(n0-n1) */
} TcMapDesc;

typedef struct {
    int32_t height, width; /* camera resolution, uniform over the handle's envs */
    int32_t obs_format;    /* TC_OBS_CLASSES or TC_OBS_RGB */
} TcSimDesc;

/* Device output pointers of a step; any pointer may be NULL to skip that output. */
typedef struct {
    uint8_t *obs;              /* see TC_OBS_*; NULL = no rendering (reference: no_observation) */
    float *cte;                /* [N] */
    float *heading_error;      /* [N] */
    float *velocity;           /* [N] */
    float *reward;             /* [N] default reward (0 when wrapped) */
    float *position;           /* [N,2] rear axle */
    float *orientation;        /* [N] */
    float *laneline_distances; /* [N,C] */
    int32_t *nearest_edge;     /* [N,C] class-local index of the nearest laneline edge (-1: empty info) */
    float *local_path;         /* [N,4,2] coordinates of the end node of each local-path edge (0 beyond path_len) */
    int32_t *local_path_nodes; /* [N,4,2] node pairs (-1 beyond path_len) */
    int32_t *path_len;         /* [N] */
    uint8_t *terminated;       /* [N] default termination (0 when wrapped) */
    uint8_t *truncated;        /* [N] */
    double *info_f64;          /* [N,4+C] float64 mirror of the scalar info (parity tests) */
    int32_t *seg_count;        /* [N,C] debug: projected segments per class */
    int32_t *seg_i32;          /* [N,sumE,4] debug: (x0,y0,x1,y1) after the int32 cast; class c starts at slot ll_edge_off[c] */
} TcOutputs;

TC_API int tc_abi_version(void);
TC_API const char *tc_last_error(void);
/* 16 hex digits: hash of the sources and compiler flags this library was built from (the loader compares it with the
 * sources next to it, so a stale prebuilt library is never used silently; benchmarks print it with their numbers). */
TC_API const char *tc_build_info(void);

TC_API int tc_create(const TcMapDesc *map, const TcSimDesc *sim, int32_t num_envs, int32_t device, TcHandle **out);
TC_API int tc_destroy(TcHandle *h);

TC_API int tc_set_car_params(TcHandle *h, const double *dev_params /*[N,TC_CP_N]*/, void *stream);
/* Handles that render small frames with one block per env (C*H*W <= 128 KB) read the rows back in this call and rebuild
 * their visible-set tables when the cameras' reach changed: the call then synchronises the stream (it is a set-up call).
 * dev_thickness: line thickness per env in 1..255, as cv2.polylines draws it; the rasteriser's 16.16 fixed-point set-up needs
 * max(H, W) + 2 * thickness < 2^15. The device array is not checked here: the Python env validates it (ValueError). */
TC_API int tc_set_camera_params(TcHandle *h, const double *dev_cam /*[N,TC_CAM_N]*/, const int32_t *dev_thickness /*[N]*/, void *stream);
/* The same with the caller's HOST copy of the rows (host_cam [N,TC_CAM_N], may be NULL): how far the cameras see decides which
 * visible-set tables the small-frame render kernels use, and with the host copy that decision needs no read-back, so the
 * call does not synchronise. Tables are built on the host once per camera reach (~50-150 ms for a map like Knuffingen) and
 * kept: returning to an earlier reach - Camera.update_params() per episode, examples/train_stanley_il.py:52-57 - costs nothing. */
TC_API int tc_set_camera_params_host(TcHandle *h, const double *dev_cam, const int32_t *dev_thickness, const double *host_cam, void *stream);
TC_API int tc_set_wrapped(TcHandle *h, int32_t wrapped); /* 1: reward 0 / terminated false (env.py:137-138) */

/* Spawn streams on the device (Map.sample_spawn's draw, map.py:61-64, under gymnasium seeding): dev_rng_state is uint64
 * [N,5] per env = PCG64 state hi, lo, increment hi, lo, buffered 32-bit half (bit 32 = valid) of
 * numpy.random.Generator(PCG64(SeedSequence(seed_i))); the host seeds it (tinycarlo_b200/pcg64.py) and the reset paths
 * advance it exactly like numpy does for choice(spawn_points) / integers(0, n_nodes-1), redrawing while the node has no
 * successor. dev_spawn_points: the config's map.spawn_points (n_spawn_points = 0: none). dev_last_spawn (optional, int32
 * [N]) receives the node of each env's most recent reset. All buffers are caller-owned and must stay alive. */
TC_API int tc_set_spawn_rng(TcHandle *h, uint64_t *dev_rng_state, const int32_t *dev_spawn_points, int32_t n_spawn_points,
                            int32_t *dev_last_spawn);

/* Next-step autoreset (gymnasium AutoresetMode.NEXT_STEP) inside tc_step: an env whose flag dev_done[i] is set is reset
 * by the step instead of being advanced (its action is ignored; reward 0, not terminated, not truncated, empty info, obs
 * of the spawn pose), drawing its spawn node from its device stream (tc_set_spawn_rng first); every step then rewrites
 * dev_done[i] = terminated | truncated. dev_done is caller-owned device memory that must stay alive; the caller may OR
 * further termination conditions (wrappers) into it between steps. NULL = off. */
TC_API int tc_set_autoreset(TcHandle *h, uint8_t *dev_done /*[N]*/);
/* Optional companion of tc_set_autoreset: every tc_step writes dev_was_reset[i] = 1 for the envs it reset instead of
 * advancing (what gymnasium's vector env reports as the autoreset step), 0 otherwise. The vectorised reward /
 * termination wrappers (tinycarlo/wrapper/reward.py, termination.py) use it to leave reset steps alone. NULL = off. */
TC_API int tc_set_reset_mask(TcHandle *h, uint8_t *dev_was_reset /*[N]*/);

/* Reset the envs with dev_mask[i] != 0 (NULL = all) to lanepath node dev_spawn_nodes[i], or - dev_spawn_nodes NULL - to a
 * node drawn from the env's device stream; renders into obs if non-NULL and zeroes their info outputs like the
 * reference's reset (car.py:47-51). */
TC_API int tc_reset(TcHandle *h, const uint8_t *dev_mask, const int32_t *dev_spawn_nodes, const TcOutputs *outs, void *stream);
TC_API int tc_step(TcHandle *h, const float *dev_car_control /*[N,2]*/, const int32_t *dev_maneuver /*[N]*/, const TcOutputs *outs, void *stream);
/* tc_step with float64 actions (the reference computes in float64 when it is fed Python floats, SURVEY H3). */
TC_API int tc_step_f64(TcHandle *h, const double *dev_car_control /*[N,2]*/, const int32_t *dev_maneuver /*[N]*/, const TcOutputs *outs, void *stream);
TC_API int tc_render(TcHandle *h, const uint8_t *dev_mask, uint8_t *dev_obs, int32_t obs_format, int32_t *dev_seg_count, int32_t *dev_seg_i32, void *stream);

TC_API int tc_get_state(TcHandle *h, double *dev_sf /*[N,TC_SF_N]*/, int32_t *dev_si /*[N,TC_SI_N]*/, void *stream);
TC_API int tc_set_state(TcHandle *h, const double *dev_sf, const int32_t *dev_si, void *stream);

/* Host-buffer step: copies the actions in, runs tc_step, copies reward/terminated/truncated/cte/heading_error back and
 * synchronises the stream. Any host output may be NULL. */
TC_API int tc_step_host(TcHandle *h, const float *host_car_control, const int32_t *host_maneuver, const TcOutputs *dev_outs,
                 float *host_reward, uint8_t *host_terminated, uint8_t *host_truncated, float *host_cte, float *host_heading_error,
                 void *stream);
/* The same, and the step's observations (dev_outs->obs, obs_bytes bytes: all envs) are copied to host_obs with ONE
 * device-to-host copy before the synchronisation - what the reference's caller holds after env.step (env.py:147 returns the
 * frame as a host array). With the 1-bit-per-pixel format (TC_OBS_CLASSES_BITS) that is 8x fewer PCIe bytes than u8 masks. */
#include <stddef.h>
TC_API int tc_step_host_obs(TcHandle *h, const float *host_car_control, const int32_t *host_maneuver, const TcOutputs *dev_outs,
                 float *host_reward, uint8_t *host_terminated, uint8_t *host_truncated, float *host_cte, float *host_heading_error,
                 void *host_obs, size_t obs_bytes, void *stream);

/* NoiseObservationWrapper (tinycarlo/wrapper/observation.py:5-33) on u8 class observations [N,C,H,W], in place: per class
 * n_blobs filled circles (centre uniform in the frame, radius uniform in [1, max_radius)), each with probability 0.3 ORs in
 * the pixels of a random class inside the circle, else erases the circle; classes ascending, blobs in sequence, like the
 * reference. The reference draws from numpy's unseeded global RNG; here the draw of (env, step, class, blob) is
 * Philox4x32-10 with key = seed and counter = (env_index_offset + env, step, class * n_blobs + blob, 0):
 * x = r0 % W, y = r1 % H, radius = 1 + r2 % (max_radius - 1), copy = (r3 & 0xffff) < 19661, source class = (r3 >> 16) % C. */
TC_API int tc_noise_blobs(TcHandle *h, uint8_t *dev_obs, uint64_t seed, uint32_t step, int32_t n_blobs, int32_t max_radius,
                          int32_t env_index_offset, const uint8_t *dev_mask, void *stream);

/* Ego-centric bird's-eye view (BEV): top-down lane masks around every car, P = C + route planes. For env i with state
 * x = sf[TC_SF_X], y = sf[TC_SF_Y], θ = sf[TC_SF_ROT] (the rear axle, in map metres; map coordinates are image-like, y down):
 *
 *   c = cos θ, s = sin θ, k = pixel_per_meter, (col0, row0) = car_pixel
 *   for a map point (px, py):  dx = px - x;  dy = py - y
 *       u = col0 + k * (dy*c - dx*s)        # car's right  -> +u (image right)
 *       v = row0 - k * (dx*c + dy*s)        # car's heading -> -v (image up)
 *
 * evaluated in float64, in exactly this order, with no FMA, then truncated with tc_np_int32 (numpy's np.int32). Plane p < C
 * is laneline class p: for every edge of that class in JSON order, cv2.polylines(plane, [[u0,v0],[u1,v1]], False, 255,
 * line_thickness) on a zero plane. With route on, plane C holds the car's tracked local path instead: the path_len lanepath
 * edges (si[2+2j], si[3+2j]) with lp_nodes coordinates, drawn the same way (what the overview draws in blue). The mapping is
 * a rotation, not a mirror: the BEV is the reference overview turned so that the car points up. */
typedef struct {
    int32_t height, width;       /* BEV resolution H, W */
    double pixel_per_meter;      /* k */
    double car_col, car_row;     /* (col0, row0): where the rear axle lands in the BEV */
    int32_t line_thickness;      /* 1..8 */
    int32_t route;               /* 1: plane C holds the tracked local path */
    int32_t format;              /* TC_OBS_CLASSES: u8 [N,P,H,W] 0/255; TC_OBS_CLASSES_BITS: u32 [N,P,H*W/32] (needs H*W % 32 == 0) */
} TcBevDesc;
/* Registers the BEV description and a caller-owned device buffer of N frames in desc->format, which must stay alive (like
 * tc_set_autoreset's buffer). From then on tc_step / tc_step_f64 re-render the BEV after the tracking kernel (one launch; it
 * reads the post-step state, so next-step autoresets need nothing extra) and tc_reset renders it for the masked envs, whether
 * or not they render the camera. dev_bev NULL switches the BEV off. */
TC_API int tc_set_bev(TcHandle *h, const TcBevDesc *desc, uint8_t *dev_bev);
/* Re-renders the BEV of the envs with dev_mask[i] != 0 (NULL = all) at the current state (after tc_set_state). */
TC_API int tc_render_bev(TcHandle *h, const uint8_t *dev_mask, void *stream);

/* Number of kernel launches issued through this handle since creation (bench.py reports it). */
TC_API int64_t tc_launch_count(const TcHandle *h);

/* Per-kernel device timing of tc_step with CUDA events recorded on the step's own stream (bench.py's roofline figure).
 * tc_profile_begin arms up to max_steps steps; tc_profile_end waits for them and returns the summed milliseconds of the
 * tracking, camera-pass and rasterise+store kernels and the number of steps recorded. */
TC_API int tc_profile_begin(TcHandle *h, int32_t max_steps);
TC_API int tc_profile_end(TcHandle *h, double *host_ms_sum /*[3]*/, int32_t *host_steps);

/* Debug hook: per-block timeline of the fused render kernel, int64 [N*C][10] = smid, clock64 at block start, tables in
 * shared memory, camera pass done, rasterisation done, stores issued, segment count, cycles zeroing / set-up / drawing. NULL switches it off. (tools/timeline.py) */
TC_API int tc_debug_set_timeline(TcHandle *h, long long *dev_timeline);

/* Debug hook: the visible-set tables of the block-per-env render kernel (small frames; tinycarlo_b200/csrc/tc_cull.h).
 * host_out4 = camera reach R in metres the tables were built for (-1: culling off, the whole laneline graph is processed;
 * -2: this handle renders per class and has no such tables), number of cell descriptors, mean and maximum node count of a
 * cell. tc_set_camera_params rebuilds the tables (and synchronises the stream) when the cameras' reach changes. Setting
 * the environment variable TC_CULL=0 switches the culling off. */
/* Episode statistics of one step in one launch (the numbers the ranks of a multi-GPU job all-gather over NCCL at log cadence):
 * dev_acc4[0] += envs with terminated | truncated, [1] += truncated, [2] += sum of rewards, [3] += n. Works on any reward / flag
 * tensors of the current device (the kernels' own outputs or what the reward / termination wrappers made of them). */
TC_API int tc_episode_stats(const float *dev_reward, const uint8_t *dev_terminated, const uint8_t *dev_truncated, int32_t n, double *dev_acc4,
                 void *stream);
TC_API int tc_debug_cull_info(TcHandle *h, double *host_out4);
/* Diagnostics: which kernels this handle launches. out8 = {block-per-env render path (0/1), envs per block of the packed
 * kernel (0: one-env kernel), its 32-segment chunks, dynamic shared memory of the render kernel, thread-per-env tracking (0/1),
 * shared memory of the banded kernel (0: unused), node capacity and table bytes of the visible-set cells}. */
/* out4 = {visible-set table builds, cache hits, host milliseconds of the last build, of all builds} */
TC_API int tc_debug_cull_stats(TcHandle *h, double *out4);
TC_API int tc_debug_render_info(TcHandle *h, int32_t *out8);

/* Test hook: the reference's Layer queries (layer.py) evaluated by the DEVICE functions on class 0 of the handle's map.
 * op: 0 get_nearest_edge(pos) 1 get_nearest_edge_with_orientation(pos, a) 2 is_position_within_edge_bounds(pos, e=(i0,i1))
 *     3 distance_to_edge(pos, e) 4 clip_angle(a).  Results: out_i[0], out_d[0] (device pointers). */
TC_API int tc_debug_layer_query(TcHandle *h, int32_t op, double px, double py, double a, int32_t i0, int32_t i1, int32_t *dev_out_i,
                         double *dev_out_d, void *stream);

#ifdef __cplusplus
}
#endif
#endif
