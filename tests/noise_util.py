"""The blob noise of NoiseObservationWrapper as a plain reference: the reference's operation (tinycarlo/wrapper/observation.py:14-27,
with cv2.circle, cv2.bitwise_and and cv2.bitwise_or) driven by the draws of the tc_noise_blobs contract in
include/tinycarlo_b200.h: Philox4x32-10 with key = seed and counter = (env, step, class * n_blobs + blob, camera), every word
reduced mod 2^32. Tests only."""
import cv2
import numpy as np

M32 = 0xFFFFFFFF


def philox4x32_10(c, k):
    """Philox4x32-10 (Random123) of the four counter words c under the two key words k"""
    c = [int(x) & M32 for x in c]
    k = [int(x) & M32 for x in k]
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k[0]) & M32, p1 & M32, ((p0 >> 32) ^ c[3] ^ k[1]) & M32, p0 & M32]
        k = [(k[0] + 0x9E3779B9) & M32, (k[1] + 0xBB67AE85) & M32]
    return c


def reference_noise(view, env_global, cam, seed, step, n_blobs, max_radius):
    """the noise of one view u8 [C, H, W] of env `env_global` (env_index_offset + local index), camera `cam`, in place;
    returns the view"""
    Cn, H, W = view.shape
    seed = int(seed) & (2**64 - 1)
    for c in range(Cn):
        for k in range(n_blobs):
            r = philox4x32_10([env_global, step, c * n_blobs + k, cam], [seed & M32, seed >> 32])
            x, y = r[0] % W, r[1] % H
            radius = 1 + r[2] % (max_radius - 1) if max_radius > 1 else 1
            if (r[3] & 0xFFFF) < 19661:
                mask = np.zeros((H, W), dtype=np.uint8)
                cv2.circle(mask, (x, y), radius, 255, -1)
                mask = cv2.bitwise_and(view[(r[3] >> 16) % Cn], mask, mask=mask)
                view[c] = cv2.bitwise_or(view[c], mask)
            else:
                cv2.circle(view[c], (x, y), radius, 0, -1)
    return view


# class count of the maps the geometry table names: tests/map_shapes_util.py's regroupings of Knuffingen and two bundled maps
CLASSES = {"K1": 1, "K2": 2, "K16": 16, "formula_student_track": 3, "knuffingen": 5}

# The geometry table: (map, envs N, cameras M, H, W, max_radius, n_blobs, seed, step, env_index_offset, mask). mask: None (no
# mask passed), "off" / "on" (all zero / all one), "random" (per env, so on a rig it selects whole envs). Radius 1023 runs on
# frames smaller than the blob on every side; the offsets put env_index_offset + env across 2^31 and, for a negative offset,
# across 2^32 (counter word 0 wraps); the rigs check counter word 3.
GEOMETRY = [
    ("knuffingen", 16, 1, 128, 160, 100, 10, 0x1234567890, 0, 0, None),
    ("knuffingen", 3, 1, 480, 640, 100, 10, 0, 7, 40, None),
    ("knuffingen", 2, 1, 1, 1, 1023, 10, 2**64 - 1, 2**32 - 1, 0, None),
    ("knuffingen", 9, 1, 84, 84, 2, 37, 0xFFFFFFFF00000000, 1, 5, "random"),
    ("knuffingen", 6, 1, 84, 84, 100, 10, 3, 2, 0, "off"),
    ("knuffingen", 6, 1, 45, 71, 100, 10, 3, 2, 0, "on"),
    ("knuffingen", 5, 1, 128, 160, 100, 0, 11, 0, 0, None),
    ("knuffingen", 10, 1, 45, 71, 3, 10, 0x1234567890, 2**32 - 1, 2**31 - 5, None),
    ("knuffingen", 4, 2, 84, 84, 1023, 2, 0, 9, 0, None),
    ("knuffingen", 8, 3, 84, 84, 100, 10, 2**64 - 1, 4, 100, "random"),
    ("K1", 8, 1, 1, 97, 1, 37, 0xFFFFFFFF00000000, 3, 0, None),
    ("K1", 8, 1, 97, 1, 2, 37, 0x1234567890, 2**32 - 1, 0, None),
    ("K1", 4, 1, 480, 640, 100, 10, 0x1234567890, 1, 2**31 - 1, None),
    ("K1", 7, 1, 84, 84, 3, 10, 0, 0, -3, "random"),
    ("K2", 6, 1, 45, 71, 3, 10, 0, 5, 0, None),
    ("K2", 3, 1, 45, 71, 1023, 10, 2**64 - 1, 0, 0, "on"),
    ("K2", 9, 2, 128, 160, 100, 37, 0xFFFFFFFF00000000, 2**32 - 1, 0, "random"),
    ("K2", 4, 1, 1, 1, 1, 37, 0x1234567890, 6, 0, None),
    ("K16", 6, 1, 84, 84, 100, 10, 0x1234567890, 0, 0, None),
    ("K16", 2, 1, 97, 1, 1023, 1, 0, 2**32 - 1, 0, None),
    ("K16", 3, 1, 128, 160, 3, 37, 2**64 - 1, 8, 0, None),
    ("K16", 2, 1, 480, 640, 2, 37, 0xFFFFFFFF00000000, 0, 0, None),
    ("K16", 5, 3, 1, 97, 100, 10, 0x1234567890, 1, 2**31 - 2, "random"),
    ("K16", 4, 1, 45, 71, 1, 10, 0, 0, 0, "off"),
    ("formula_student_track", 20, 1, 84, 84, 100, 10, 0x1234567890, 3, 0, "random"),
    ("formula_student_track", 8, 1, 1, 1, 1, 37, 2**64 - 1, 2**32 - 1, 0, None),
    ("formula_student_track", 3, 1, 45, 71, 1023, 1, 0xFFFFFFFF00000000, 0, 0, None),
    ("formula_student_track", 6, 1, 97, 1, 100, 0, 0, 0, 0, "on"),
    ("formula_student_track", 5, 2, 480, 640, 100, 10, 0, 2, 7, None),
    ("formula_student_track", 4, 3, 128, 160, 2, 37, 0x1234567890, 2**32 - 1, 0, "on"),
]


def geometry_id(row):
    mp, N, M, H, W, r, nb, seed, step, off, mask = row
    return f"{mp}-{N}x{M}-{H}x{W}-r{r}-b{nb}-s{seed:x}-t{step:x}-o{off}-{mask}"


def make_mask(kind, N, rng):
    """the per-env mask of a geometry row (uint8 [N] or None); "random" selects at least one env and leaves at least one out"""
    if kind is None:
        return None
    if kind == "random":
        m = rng.integers(0, 2, N).astype(np.uint8)
        m[0], m[-1] = 1, 0
        return m
    return np.full(N, 1 if kind == "on" else 0, np.uint8)


def expected_noise(obs, row, mask, views=None):
    """reference_noise applied to the views of obs u8 [N, M, C, H, W] (a copy) that the mask selects; views: the env indices to
    compute (default all), the others come back as they were"""
    mp, N, M, H, W, r, nb, seed, step, off, _ = row
    out = obs.copy()
    for i in range(N) if views is None else views:
        if mask is not None and not mask[i]:
            continue
        for m in range(M):
            reference_noise(out[i, m], (off + i) & M32, m, seed, step, nb, r)
    return out
