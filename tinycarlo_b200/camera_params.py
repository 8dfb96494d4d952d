"""Extrinsic / intrinsic camera matrices on the host (tinycarlo/camera.py:145-178).

E = Rodrigues([pitch-90, roll, 0] deg) @ Rodrigues([0, 0, yaw+90] deg) @ [I | -position];  K from fov and resolution.
For bit parity the same cv2.Rodrigues / numpy calls as the reference are used (a textbook Rodrigues agrees to 3e-16 but
not bit for bit, SURVEY H10). These run only at construction / parameter change, never per step."""
import numpy as np

from . import _rodrigues


def extrinsic_matrix(position, orientation) -> np.ndarray:
    angles_rad = np.radians(np.asarray(orientation) + np.array([-90, 0, 90]))
    rotation_matrix_pr = _rodrigues.rodrigues(np.array([1, 1, 0]) * angles_rad)
    rotation_matrix_y = _rodrigues.rodrigues(np.array([0, 0, 1]) * angles_rad)
    translation_matrix = np.column_stack((np.eye(3), -np.array(position)))
    return np.asarray(rotation_matrix_pr @ rotation_matrix_y @ translation_matrix, np.float64)


def intrinsic_matrix(fov_deg, resolution) -> np.ndarray:
    fov_radians = np.radians(fov_deg)
    fx = resolution[1] / (2 * np.tan(fov_radians / 2))
    fy = resolution[0] / (2 * np.tan(fov_radians / 2))
    return np.array([[fx, 0, resolution[1] / 2], [0, fy, resolution[0] / 2], [0, 0, 1]], np.float64)


def camera_row(position, orientation, fov, resolution, max_range) -> np.ndarray:
    """One row of the per-env camera table (include/tinycarlo_b200.h TC_CAM_*)."""
    E = extrinsic_matrix(position, orientation)
    K = intrinsic_matrix(fov, resolution)
    row = np.zeros(20, np.float64)
    row[:12] = E.reshape(-1)
    row[12], row[13], row[14], row[15] = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    row[16] = float(max_range)
    return row


def view_rows(cam_cfgs, n_envs: int):
    """Camera rows [n_envs*M, 20] and line thicknesses int32 [n_envs*M] for M camera sections (config.camera_params), one per
    view in env-major order: view v = env * M + m has camera m (include/tinycarlo_b200.h tc_create_rig)."""
    rows = np.stack([camera_row(c["position"], c["orientation"], c["fov"], c["resolution"], c["max_range"]) for c in cam_cfgs])
    thickness = np.array([int(c["line_thickness"]) for c in cam_cfgs], np.int32)
    return np.tile(rows, (n_envs, 1)), np.tile(thickness, n_envs)
