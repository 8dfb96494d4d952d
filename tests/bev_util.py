"""The bird's-eye-view contract (include/tinycarlo_b200.h, tc_set_bev) restated in numpy + cv2.polylines: the oracle the
host build (tests/test_bev_host.py) and the device kernel (tests/test_gpu_bev.py) are compared against, and the binding of
the host build's ht_bev."""
import ctypes as C
import math

import numpy as np


def bev_points(pts, x, y, c, s, k, col0, row0):
    """map points [m,2] -> int32 BEV pixels [m,2], float64 in the contract's order, truncated like np.int32"""
    pts = np.asarray(pts, np.float64).reshape(-1, 2)
    dx = pts[:, 0] - x
    dy = pts[:, 1] - y
    u = col0 + k * (dy * c - dx * s)
    v = row0 - k * (dx * c + dy * s)
    with np.errstate(invalid="ignore"):
        return np.stack([u, v], -1).astype(np.int32)


def oracle_bev(tables, sf_row, si_row, H, W, pixel_per_meter, car_pixel, thickness, route=False, cs=None):
    """u8 [P,H,W] of one env. cs: (cos, sin) of the heading to use instead of libm's (the device's may differ by an ulp)."""
    import cv2
    x, y, rot = float(sf_row[0]), float(sf_row[1]), float(sf_row[2])
    c, s = cs if cs is not None else (math.cos(rot), math.sin(rot))
    col0, row0 = float(car_pixel[0]), float(car_pixel[1])
    C = tables.n_classes
    out = np.zeros((C + int(bool(route)), H, W), np.uint8)

    def draw(p, nodes, edges):
        # one 2-point polyline per edge; drawn in one call, which ORs the same pixels as one call per edge (one colour)
        edges = np.asarray(edges, np.int64).reshape(-1, 2)
        if len(edges):
            uv = bev_points(nodes, x, y, c, s, pixel_per_meter, col0, row0)
            cv2.polylines(out[p], np.ascontiguousarray(uv[edges]), False, 255, int(thickness))
    for cl in range(C):
        draw(cl, tables.class_nodes(cl), tables.class_edges(cl))
    if route:
        n = min(max(int(si_row[0]), 0), 4)
        draw(C, tables.lp_nodes, [(int(si_row[2 + 2 * j]), int(si_row[3 + 2 * j])) for j in range(n)])
    return out


def oracle_bev_ulp(tables, sf_row, si_row, got, bits=False, **kw):
    """Compares a device BEV frame with the oracle (bits: `got` is the classes_bits frame, compared with pack_bits of the
    oracle's). -> 0: identical with libm's cos / sin, 1: identical once cos or sin is moved by one ulp (the documented
    device-versus-glibc difference), -1: anything else."""
    def same(cs=None):
        want = oracle_bev(tables, sf_row, si_row, cs=cs, **kw)
        return np.array_equal(got, pack_bits(want) if bits else want)
    if same():
        return 0
    rot = float(sf_row[2])
    c, s = math.cos(rot), math.sin(rot)
    for cc in (np.nextafter(c, -np.inf), c, np.nextafter(c, np.inf)):
        for ss in (np.nextafter(s, -np.inf), s, np.nextafter(s, np.inf)):
            if (cc, ss) != (c, s) and same((float(cc), float(ss))):
                return 1
    return -1


def pack_bits(u8):
    """u8 0/255 [..., P, H, W] -> int32 [..., P, H*W/32]: bit (y*W+x)%32 of word (y*W+x)/32 is pixel (x, y)"""
    b = (np.asarray(u8) != 0).reshape(u8.shape[:-2] + (-1,))
    return np.packbits(b, axis=-1, bitorder="little").view(np.int32)


def host_bev(core, sf, si, H, W, pixel_per_meter, car_pixel, thickness, route=False):
    """ht_bev (tc_hosttest.cpp): the BEV of n envs at state rows sf [n,8] / si [n,16] through the host build of tc_core.cuh, for the
    map of `core` (a hosttest_util.HostCore) -> u8 [n,P,H,W]"""
    from hosttest_util import P, ht
    from tinycarlo_b200 import _lib
    L = ht()
    L.ht_bev.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(_lib.TcBevDesc), C.c_void_p]
    sf = np.ascontiguousarray(sf, np.float64).reshape(-1, 8)
    si = np.ascontiguousarray(si, np.int32).reshape(-1, 16)
    n = len(sf)
    out = np.zeros((n, core.C + int(bool(route)), H, W), np.uint8)
    d = _lib.TcBevDesc(H, W, float(pixel_per_meter), float(car_pixel[0]), float(car_pixel[1]), int(thickness), int(bool(route)), 0)
    L.ht_bev(core.h, n, P(sf), P(si), C.byref(d), P(out))
    return out
