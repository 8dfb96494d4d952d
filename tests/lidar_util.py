"""The range-scan contract (include/tinycarlo_b200.h, tc_set_lidar) restated in numpy: the oracle the host build
(tests/test_lidar_host.py) and the device kernel (tests/test_gpu_lidar.py) are compared against, and the binding of the host
build's ht_lidar."""
import ctypes as C
import math

import numpy as np


def ray_ab(rays, fov):
    """(cos phi_j, sin phi_j) [R,2] of the contract's ray angles, with the host libm (what tc_set_lidar uploads)"""
    ab = np.zeros((rays, 2))
    for j in range(rays):
        phi = (fov * ((j + 0.5) / rays) - fov / 2) * (math.pi / 180)
        ab[j] = math.cos(phi), math.sin(phi)
    return ab


def oracle_lidar(tables, sf_row, rays, fov, max_range, origin=(0.0, 0.0), cs=None):
    """float64 [C,R] of one env, before the float32 cast. cs: (cos, sin) of the heading to use instead of libm's (the device's
    may differ by an ulp)."""
    x, y, rot = float(sf_row[0]), float(sf_row[1]), float(sf_row[2])
    c, s = cs if cs is not None else (math.cos(rot), math.sin(rot))
    f, r = float(origin[0]), float(origin[1])
    ox = x + (f * c - r * s)
    oy = y + (f * s + r * c)
    ab = ray_ab(rays, fov)
    a, b = ab[:, 0], ab[:, 1]
    dx = (a * c - b * s)[:, None]
    dy = (a * s + b * c)[:, None]
    out = np.full((tables.n_classes, rays), float(max_range))
    for p in range(tables.n_classes):
        nodes, edges = tables.class_nodes(p), np.asarray(tables.class_edges(p), np.int64).reshape(-1, 2)
        if not len(edges):
            continue
        A, B = nodes[edges[:, 0]], nodes[edges[:, 1]]
        ex, ey = (B[:, 0] - A[:, 0])[None], (B[:, 1] - A[:, 1])[None]
        wx, wy = (A[:, 0] - ox)[None], (A[:, 1] - oy)[None]
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            den = dx * ey - dy * ex
            t = (wx * ey - wy * ex) / den
            u = (wx * dy - wy * dx) / den
            hit = (den != 0) & (t >= 0) & (u >= 0) & (u <= 1)
        out[p] = np.minimum(float(max_range), np.where(hit, t, np.inf).min(1))
    out[out == 0] = 0.0   # a zero distance is +0.0
    return out


def f32_bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def oracle_lidar_ulp(tables, sf_row, got, **kw):
    """Compares a device scan (float32 [C,R]) with the oracle's float32 cast, bit pattern for bit pattern. -> 0: identical with
    libm's cos / sin, 1: identical once cos or sin is moved by one ulp (the documented device-versus-glibc difference),
    -1: anything else."""
    g = f32_bits(got)

    def same(cs=None):
        return np.array_equal(g, f32_bits(oracle_lidar(tables, sf_row, cs=cs, **kw)))
    if same():
        return 0
    rot = float(sf_row[2])
    c, s = math.cos(rot), math.sin(rot)
    for cc in (np.nextafter(c, -np.inf), c, np.nextafter(c, np.inf)):
        for ss in (np.nextafter(s, -np.inf), s, np.nextafter(s, np.inf)):
            if (cc, ss) != (c, s) and same((float(cc), float(ss))):
                return 1
    return -1


def host_lidar(core, sf, rays, fov, max_range, origin=(0.0, 0.0)):
    """ht_lidar (tc_hosttest.cpp): the scan of n envs at state rows sf [n,8] through the host build of tc_core.cuh, for the map
    of `core` (a hosttest_util.HostCore) -> float64 [n,C,R]"""
    from hosttest_util import P, ht
    from tinycarlo_b200 import _lib
    L = ht()
    L.ht_lidar.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(_lib.TcLidarDesc), C.c_void_p]
    sf = np.ascontiguousarray(sf, np.float64).reshape(-1, 8)
    n = len(sf)
    out = np.zeros((n, core.C, rays))
    d = _lib.TcLidarDesc(int(rays), float(fov), float(max_range), float(origin[0]), float(origin[1]))
    L.ht_lidar(core.h, n, P(sf), C.byref(d), P(out))
    return out


def host_keep(desc, o, cs, a, b):
    """ht_lidar_keep: does the cull (tc_lidar_stage) keep edge (a, b) for origin o and heading (cos, sin) cs?"""
    from hosttest_util import ht
    L = ht()
    L.ht_lidar_keep.argtypes = [C.c_void_p] + [C.c_double] * 8
    return bool(L.ht_lidar_keep(C.byref(desc), *(float(v) for v in (o[0], o[1], cs[0], cs[1], a[0], a[1], b[0], b[1]))))


# The synthetic map of the exact cases (pixel_per_meter 1: nodes in metres). With the car at (0, 0) heading +x (rot 0) and an
# odd number of rays over any fov, ray (R-1)/2 is exactly (1, 0); with max_range SYN_RANGE = 0.25 (exactly representable):
SYN_RANGE = 0.25
_SUCC = float(np.nextafter(SYN_RANGE, np.inf))
SYN_LAYERS = {
    "u0": ([[0.2, 0.0], [0.2, 0.3]], [[0, 1]]),           # the forward ray meets it at u = 0 exactly, t = 0.2
    "u1": ([[0.15, -0.3], [0.15, 0.0]], [[0, 1]]),        # at u = 1 exactly, t = 0.15
    "zero": ([[0.0, -0.1], [0.0, 0.1]], [[0, 1]]),        # through the car: t = 0 (stored +0.0) on every ray not along it
    "parallel": ([[0.05, 0.05], [0.2, 0.05]], [[0, 1]]),  # parallel to the forward ray, beside it
    "collinear": ([[0.05, 0.0], [0.2, 0.0]], [[0, 1]]),   # on the forward ray: den == 0, never hits
    "point": ([[0.1, 0.0]], [[0, 0]]),                   # zero length, on the forward ray
    "at_range": ([[SYN_RANGE, -0.1], [SYN_RANGE, 0.1]], [[0, 1]]),   # t = max_range
    "beyond": ([[_SUCC, -0.1], [_SUCC, 0.1]], [[0, 1]]),             # one ulp beyond max_range
    "crossing": ([[0.1, -5.0], [0.1, 5.0]], [[0, 1]]),   # crosses the cull's square, both ends far outside it
    # u near 1 by an ulp either way: den = RN(k * 1e-17 - 0.2) is -0.2 or a neighbour, un = -0.2
    **{f"near1_{k}": ([[0.12, 0.2], [0.12, k * 1e-17]], [[0, 1]]) for k in (-3, -2, 2, 3)},
}


def synthetic_map(directory):
    """writes the synthetic map to `directory` -> its path"""
    import json
    import os
    data = {"width": 100, "height": 100,
            "lanelines": {k: {"layer_color": [(40 * i) % 256, 255 - (15 * i) % 256, 100], "nodes": nodes, "edges": edges}
                          for i, (k, (nodes, edges)) in enumerate(SYN_LAYERS.items())},
            "lanepath": {"layer_color": [0, 0, 255], "nodes": [[-5.0, 0.0], [-4.0, 0.0], [-3.0, 0.0]], "edges": [[0, 1], [1, 2]]}}
    path = os.path.join(str(directory), "lidar_synthetic.json")
    with open(path, "w") as f:
        json.dump(data, f)
    return path
