"""CPU tests of the blob noise (tc_noise_blobs, NoiseObservationWrapper) through the host build of its arithmetic: the Philox
draw, the midpoint-circle table and the kernel's fill, replayed sequentially by ht_noise_blobs (tc_hosttest.cpp) from the same
tc_core.cuh helpers the kernel calls. The yardsticks are the published Philox4x32-10 vectors, cv2.circle and the reference's
operation (tests/noise_util.py)."""
import zlib

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from hosttest_util import circle, noise_blobs, philox  # noqa: E402
from noise_util import CLASSES, GEOMETRY, expected_noise, geometry_id, make_mask, philox4x32_10  # noqa: E402

M32 = 0xFFFFFFFF

# Random123's known-answer vectors for philox4x32_10 (kat_vectors): counter, key, result
KATS = [
    ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
    ([M32] * 4, [M32] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
]


@pytest.mark.parametrize("ctr,key,want", KATS, ids=["zero", "ones", "pi"])
def test_philox_known_answers(ctr, key, want):
    assert philox4x32_10(ctr, key) == want
    assert philox(np.array([ctr]), np.array([key]))[0].tolist() == want


def test_philox_host_build_matches_the_model():
    """10^4 counters and keys: uniform words, words drawn from {0, 2^32 - 1, uniform}, and every word alone at 0 and 2^32 - 1"""
    rng = np.random.default_rng(7)
    n = 10000
    words = rng.integers(0, 2**32, (n, 6), dtype=np.uint64)
    pick = rng.integers(0, 3, (n, 6))
    mixed = slice(n // 2, n)
    words[mixed] = np.where(pick[mixed] == 0, 0, np.where(pick[mixed] == 1, M32, words[mixed]))
    for j in range(6):
        words[2 * j, j], words[2 * j + 1, j] = 0, M32
    words = words.astype(np.uint32)
    got = philox(words[:, :4], words[:, 4:])
    want = np.array([philox4x32_10(w[:4], w[4:]) for w in words.tolist()], np.uint32)
    assert np.array_equal(got, want)


def cv2_disc(H, W, centre, radius):
    img = np.zeros((H, W), np.uint8)
    cv2.circle(img, (int(centre[0]), int(centre[1])), int(radius), 255, -1)
    return img


def test_circle_matches_cv2_at_every_radius():
    """the disc of tc_circle_halfwidths through the kernel's fill equals cv2.circle(..., -1) for every radius the ABI accepts
    (1..1022: max_radius <= 1023 draws radius <= 1022), at an interior centre off the frame's diagonal"""
    for r in range(1, 1023):
        H, W, centre = 2 * r + 3, 2 * r + 6, (r + 4, r + 1)
        assert np.array_equal(circle(H, W, centre, r), cv2_disc(H, W, centre, r)), r


@pytest.mark.parametrize("H,W", [(1, 1), (1, 97), (97, 1), (45, 71), (84, 84), (480, 640)])
def test_circle_clipped_matches_cv2(H, W):
    """centres anywhere in the frame (as the draws place them), radii from 1 to past every side: clipped on 0 to 4 sides"""
    rng = np.random.default_rng(H * 1000 + W)
    radii = np.concatenate([[1, 2, 3, 1022], rng.integers(1, max(H, W) + 2, 150), rng.integers(1, 1023, 30)])
    sides = set()
    for r in radii.tolist():
        x, y = int(rng.integers(0, W)), int(rng.integers(0, H))
        assert np.array_equal(circle(H, W, (x, y), r), cv2_disc(H, W, (x, y), r)), (x, y, r)
        sides.add((x - r < 0) + (x + r >= W) + (y - r < 0) + (y + r >= H))
    assert 4 in sides and (min(H, W) < 3 or 0 in sides)


@pytest.mark.parametrize("row", GEOMETRY, ids=[geometry_id(r) for r in GEOMETRY])
def test_host_noise_matches_the_reference_operation(row):
    """ht_noise_blobs equals the reference's operation byte for byte on random bytes (not 0/255 masks), so that every OR
    and every erase shows"""
    mp, N, M, H, W, r, nb, seed, step, off, mask_kind = row
    rng = np.random.default_rng(zlib.crc32(geometry_id(row).encode()))
    obs = rng.integers(0, 256, (N, M, CLASSES[mp], H, W), dtype=np.uint8)
    mask = make_mask(mask_kind, N, rng)
    got = noise_blobs(obs, seed, step, nb, r, off, mask)
    want = expected_noise(obs, row, mask)
    for i in range(N):
        assert np.array_equal(got[i], want[i]), i
    if nb == 0 or mask_kind == "off":
        assert np.array_equal(got, obs)
    else:
        assert not np.array_equal(got, obs)
