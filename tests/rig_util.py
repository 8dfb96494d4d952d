"""Camera-rig helpers of the tests: the host build's tracking step with M cameras per env (ht_track_rig in
tinycarlo_b200/csrc/tc_hosttest.cpp) and the oracle's frame of one view. View v = i * M + m is camera m of env i."""
import ctypes as C

import numpy as np

import hosttest_util as HU
from oracle import oracle as orc

REAR = {"orientation": [22, 0, 180]}   # the shipped pitch, looking backwards


def ht_rig():
    L = HU.ht()
    L.ht_track_rig.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 14
    return L


class HostRig(HU.HostCore):
    """HostCore with M cameras per env: cam [n*M,20], pose [n*M,12] and the reset's view mask [n*M] (tracking only)."""

    def __init__(self, tables, n, n_cams, car_rows, cam_rows, thickness, H, W):
        super().__init__(tables, n, car_rows, np.asarray(cam_rows)[:1], np.asarray(thickness).reshape(-1)[:1], H, W)
        self.M = n_cams
        self.cam = np.ascontiguousarray(np.asarray(cam_rows, np.float64).reshape(n * n_cams, 20))
        self.thick = np.array(np.broadcast_to(np.asarray(thickness, np.int32).reshape(-1), (n * n_cams,)), order="C")
        self.pose = np.zeros((n * n_cams, 12))
        self.view_mask = np.full(n * n_cams, 0xEE, np.uint8)

    def _track(self, mode, cc, man, mask, spawn):
        P = HU.P
        ht_rig().ht_track_rig(self.h, self.n, self.M, mode, self.wrapped, P(self.sf), P(self.si), P(self.car), P(self.cam), P(self.pose),
                              P(cc), P(man), P(mask), P(spawn), P(self.info), P(self.nearest), P(self.terminated), P(self.truncated),
                              P(self.view_mask))


def oracle_pose(cam_row, sf_row):
    """orc_camera_pose: the pose of a camera row at a car state"""
    pose = np.zeros(12)
    orc.lib().orc_camera_pose(orc._p(np.ascontiguousarray(cam_row, np.float64), orc._dp), orc._p(np.ascontiguousarray(sf_row, np.float64), orc._dp),
                              orc._p(pose, orc._dp))
    return pose


def oracle_views(omap, cam_rows, thickness, sf, n_cams, H, W, fmt, views=None):
    """orc_capture_frame of view v (camera row v, thickness v, state of env v // n_cams) for every view (or those listed):
    u8 [V,C,H,W] masks or [V,H,W,3] RGB"""
    rgb = fmt == "rgb"
    V = len(cam_rows)
    out = np.zeros((V,) + ((H, W, 3) if rgb else (omap.C, H, W)), np.uint8)
    for v in range(V) if views is None else views:
        orc.lib().orc_capture_frame(omap.handle, orc._p(np.ascontiguousarray(cam_rows[v], np.float64), orc._dp), H, W, int(thickness[v]),
                                    orc._p(omap.colors, orc._up), orc._p(np.ascontiguousarray(sf[v // n_cams], np.float64), orc._dp),
                                    1 if rgb else 0, orc._p(out[v], orc._up), None, None, None, None)
    return out


def oracle_view_segments(omap, cam_row, thickness, sf_row, H, W):
    """projected segments of one view: (count[C], seg_i32[sumE,4])"""
    C_, ne = omap.C, int(omap.edge_off[-1])
    cnt = np.zeros(C_, np.int32)
    s32 = np.zeros((max(ne, 1), 4), np.int32)
    s64 = np.zeros((max(ne, 1), 4), np.float64)
    se = np.full(max(ne, 1), -1, np.int32)
    orc.lib().orc_capture_frame(omap.handle, orc._p(np.ascontiguousarray(cam_row, np.float64), orc._dp), H, W, int(thickness),
                                orc._p(omap.colors, orc._up), orc._p(np.ascontiguousarray(sf_row, np.float64), orc._dp), 0, None,
                                orc._p(cnt, orc._ip), orc._p(s32, orc._ip), orc._p(s64, orc._dp), orc._p(se, orc._ip))
    return cnt, s32
