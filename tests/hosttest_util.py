"""Builds and binds libtc_hosttest.so: the CPU-only TEST build of the kernel arithmetic (tinycarlo_b200/csrc/tc_core.cuh
compiled by g++ with one lane per group). Tests only; the product never loads it."""
import ctypes as C
import os
import subprocess

import numpy as np

from tinycarlo_b200 import _lib
from tinycarlo_b200.maptables import MapTables

HT_PATH = os.path.join(_lib.LIB_DIR, "libtc_hosttest.so")
SRC = os.path.join(_lib.CSRC, "tc_hosttest.cpp")


def build():
    deps = [SRC] + [os.path.join(_lib.CSRC, f) for f in ("tc_core.cuh", "tc_pack.h", "tc_cull.h")]
    if not os.path.exists(HT_PATH) or os.path.getmtime(HT_PATH) < max(os.path.getmtime(d) for d in deps):
        os.makedirs(_lib.LIB_DIR, exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fvisibility=hidden", "-shared", "-x", "c++",
                               "-o", HT_PATH, SRC, "-lm"])
    return HT_PATH


_ht = None


def ht():
    global _ht
    if _ht is None:
        L = C.CDLL(build())
        vp, i = C.c_void_p, C.c_int
        L.ht_map_create.restype = vp
        L.ht_map_create.argtypes = [C.POINTER(_lib.TcMapDesc)]
        L.ht_map_destroy.argtypes = [vp]
        L.ht_track.argtypes = [vp, i, i, i] + [vp] * 13
        L.ht_render.argtypes = [vp, i, i, i, i, i] + [vp] * 7
        L.ht_spawn_draws.argtypes = [vp, i, vp, vp, i, i, vp]
        L.ht_pcg_bounded.argtypes = [i, vp, C.c_uint32, i, vp]
        L.ht_cull_create.restype = vp
        L.ht_cull_create.argtypes = [C.POINTER(_lib.TcMapDesc), C.c_double, C.c_double, C.c_double]
        L.ht_cull_destroy.argtypes = [vp]
        L.ht_cull_info.argtypes = [vp, vp]
        L.ht_cull_radius_of.restype = C.c_double
        L.ht_cull_radius_of.argtypes = [vp, i, i]
        L.ht_project_culled.argtypes = [vp, vp, i, i, i, vp, vp, vp, vp, vp]
        L.ht_nearest.argtypes = [vp, i, vp, i, i, vp, vp, vp]
        L.ht_polyline.argtypes = [vp, i, i, C.c_int32, C.c_int32, C.c_int32, C.c_int32, i, i, i, i]
        L.ht_philox.argtypes = [i, vp, vp, vp]
        L.ht_circle.argtypes = [vp, i, i, i, i, i]
        L.ht_noise_blobs.argtypes = [vp, i, i, i, i, i, C.c_uint64, C.c_uint32, i, i, C.c_int32, vp]
        _ht = L
    return _ht


def P(a):
    return None if a is None else a.ctypes.data


class HostCore:
    """n envs through the host build of the kernel arithmetic, same array layouts as the C ABI."""

    def __init__(self, tables: MapTables, n, car_rows, cam_rows, thickness, H, W, fmt="classes", wrapped=False, rows_per_band=0):
        m = tables
        self.keep = [np.ascontiguousarray(a) for a in (m.ll_node_off, m.ll_edge_off, m.ll_nodes, m.ll_edges, m.colors, m.lp_nodes,
                                                      m.lp_edges, m.lp_orient, m.lp_orient_rev)]
        k = self.keep
        desc = _lib.TcMapDesc(m.n_classes, P(k[0]), P(k[1]), P(k[2]), P(k[3]), P(k[4]), len(m.lp_nodes), len(m.lp_edges), P(k[5]),
                              P(k[6]), P(k[7]), P(k[8]))
        self.desc = desc
        self.h = ht().ht_map_create(C.byref(desc))
        assert self.h
        self.n, self.H, self.W, self.C = n, H, W, m.n_classes
        self.fmt = 0 if fmt == "classes" else 1
        self.wrapped = int(wrapped)
        self.rows_per_band = rows_per_band
        self.car = np.array(np.broadcast_to(np.asarray(car_rows, np.float64).reshape(-1, 8), (n, 8)), order="C")
        self.cam = np.array(np.broadcast_to(np.asarray(cam_rows, np.float64).reshape(-1, 20), (n, 20)), order="C")
        self.thick = np.array(np.broadcast_to(np.asarray(thickness, np.int32).reshape(-1), (n,)), order="C")
        self.sf = np.zeros((n, 8))
        self.si = np.full((n, 16), -1, np.int32)
        self.pose = np.zeros((n, 12))
        self.info = np.zeros((n, 4 + self.C))
        self.nearest = np.full((n, self.C), -1, np.int32)
        self.terminated = np.zeros(n, np.uint8)
        self.truncated = np.zeros(n, np.uint8)
        sumE = int(m.ll_edge_off[-1])
        self.seg = np.zeros((n, max(sumE, 1), 4), np.int32)
        self.seg_count = np.zeros((n, self.C), np.int32)
        self.obs = np.zeros((n, self.C, H, W) if self.fmt == 0 else (n, H, W, 3), np.uint8)

    def _track(self, mode, cc, man, mask, spawn):
        ht().ht_track(self.h, self.n, mode, self.wrapped, P(self.sf), P(self.si), P(self.car), P(self.cam), P(self.pose), P(cc), P(man),
                      P(mask), P(spawn), P(self.info), P(self.nearest), P(self.terminated), P(self.truncated))

    def render(self, mask=None):
        ht().ht_render(self.h, self.n, self.H, self.W, self.fmt, self.rows_per_band, P(self.pose), P(self.cam), P(self.thick), P(mask),
                       P(self.obs), P(self.seg_count), P(self.seg))

    def project_culled(self, radius, cell=0.25, margin=0.05):
        """segments of the current poses through the visible-set tables built for camera reach `radius` ->
        (seg_count [n,C], seg [n,sumE,4], nodes of each env's cell, table info)"""
        hc = ht().ht_cull_create(C.byref(self.desc), float(radius), float(cell), float(margin))
        cnt = np.zeros_like(self.seg_count)
        seg = np.zeros_like(self.seg)
        cell_nodes = np.zeros(self.n, np.int32)
        info = np.zeros(6)
        ht().ht_project_culled(self.h, hc, self.n, self.H, self.W, P(self.pose), P(self.cam), P(cnt), P(seg), P(cell_nodes))
        ht().ht_cull_info(hc, P(info))
        ht().ht_cull_destroy(hc)
        return cnt, seg, cell_nodes, info

    def reset(self, spawn_nodes, mask=None, render=True):
        sp = np.ascontiguousarray(spawn_nodes, np.int32)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self._track(1, None, None, m, sp)
        if render:
            self.render(m)

    def step(self, cc, man, render=True):
        cc = np.ascontiguousarray(cc, np.float32).reshape(self.n, 2)
        man = np.ascontiguousarray(man, np.int32).reshape(self.n)
        self._track(0, cc, man, None, None)
        if render:
            self.render()


def philox(ctr, key):
    """Philox4x32-10 of counters ctr [n,4] under keys key [n,2] (uint32) -> [n,4]"""
    ctr, key = np.ascontiguousarray(ctr, np.uint32), np.ascontiguousarray(key, np.uint32)
    out = np.zeros((len(ctr), 4), np.uint32)
    ht().ht_philox(len(ctr), P(ctr), P(key), P(out))
    return out


def circle(H, W, centre, radius):
    img = np.zeros((H, W), np.uint8)
    ht().ht_circle(P(img), H, W, int(centre[0]), int(centre[1]), int(radius))
    return img


def noise_blobs(obs, seed, step, n_blobs, max_radius, env_index_offset=0, mask=None):
    """ht_noise_blobs on obs u8 [N, M, C, H, W] (a copy), mask per env -> the noised copy"""
    out = np.array(obs, np.uint8, order="C")
    N, M, Cn, H, W = out.shape
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    ht().ht_noise_blobs(P(out), N, M, Cn, H, W, int(seed) & (2**64 - 1), int(step) & 0xFFFFFFFF, int(n_blobs), int(max_radius),
                        int(env_index_offset), P(m))
    return out


def polyline(H, W, p0, p1, t, y_lo=0, y_hi=0, nlanes=1):
    img = np.zeros((H, W), np.uint8)
    ht().ht_polyline(P(img), H, W, int(p0[0]), int(p0[1]), int(p1[0]), int(p1[1]), int(t), y_lo, y_hi, nlanes)
    return img
