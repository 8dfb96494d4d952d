"""Vectorised PCG64 streams, bit-compatible with numpy.random.Generator(PCG64(SeedSequence(seed))) for the two draws the
reference's spawn sampling makes (tinycarlo/map.py:61): Generator.choice(list) and Generator.integers(0, n).

One numpy Generator per env costs ~4 us per scalar draw in the interpreter; a vector env with 16384 envs pre-draws
10^5..10^6 spawn nodes, so the three ingredients are restated here on numpy arrays (one lane per env):

  * SeedSequence(entropy).generate_state(4, uint64) — the hashmix / mix pool of numpy/random/bit_generator.pyx
  * PCG64: 128-bit LCG `state = state * 0x2360ED051FC65DA44385DF649FCCF645 + inc`, output XSL-RR 128/64, seeded by
    pcg64_srandom(initstate = s0<<64|s1, initseq = s2<<64|s3), with the bit generator's buffered next_uint32
  * bounded integers below 2^32: Lemire's multiply-shift with rejection (buffered_bounded_lemire_uint32)

tests/test_host_logic.py checks the streams against numpy itself (thousands of seeds, ranges that exercise the rejection
loop) and against the spawn draws recorded from the reference."""
from typing import Optional, Tuple

import numpy as np

_U32 = np.uint32
_U64 = np.uint64
_M32 = _U64(0xFFFFFFFF)

INIT_A, MULT_A = _U32(0x43B0D7E5), _U32(0x931E8875)
INIT_B, MULT_B = _U32(0x8B51F9DD), _U32(0x58F38DED)
MIX_MULT_L, MIX_MULT_R = _U32(0xCA01F9DD), _U32(0x4973F715)
XSHIFT = _U32(16)
PCG_MULT_HI, PCG_MULT_LO = _U64(0x2360ED051FC65DA4), _U64(0x4385DF649FCCF645)


def _hashmix(value, hash_const):
    value = value ^ hash_const
    hash_const = hash_const * MULT_A
    value = value * hash_const
    value = value ^ (value >> XSHIFT)
    return value, hash_const


def _mix(x, y):
    r = MIX_MULT_L * x - MIX_MULT_R * y
    return r ^ (r >> XSHIFT)


def seed_sequence_state(seeds: np.ndarray, spawn_key: Tuple[int, ...] = ()) -> np.ndarray:
    """SeedSequence(int(seed), spawn_key=spawn_key).generate_state(4, np.uint64) for every non-negative seed < 2^64 -> uint64
    [n, 4]. spawn_key (words < 2^32) is what SeedSequence.spawn gives its children: spawn(1)[0] has spawn_key (0,). numpy pads
    the seed's words to the pool size of 4 and mixes every word beyond the pool into all pool words ("remaining entropy")."""
    key = [int(k) for k in spawn_key]
    assert all(0 <= k <= 0xFFFFFFFF for k in key)
    with np.errstate(over="ignore"):
        seeds = np.asarray(seeds, dtype=_U64)
        n = len(seeds)
        lo, hi = (seeds & _M32).astype(_U32), (seeds >> _U64(32)).astype(_U32)
        two_words = hi != 0                         # entropy is the little-endian uint32 words of the integer
        pool = np.zeros((4, n), _U32)
        hc = np.full(n, INIT_A, _U32)
        ent = [lo, np.where(two_words, hi, _U32(0)), np.zeros(n, _U32), np.zeros(n, _U32)]
        for i in range(4):
            pool[i], hc = _hashmix(ent[i].copy(), hc)
        for i_src in range(4):
            for i_dst in range(4):
                if i_src != i_dst:
                    h, hc = _hashmix(pool[i_src].copy(), hc)
                    pool[i_dst] = _mix(pool[i_dst], h)
        for word in key:
            for i_dst in range(4):
                h, hc = _hashmix(np.full(n, word, _U32), hc)
                pool[i_dst] = _mix(pool[i_dst], h)
        out = np.zeros((8, n), _U32)
        hc = np.full(n, INIT_B, _U32)
        for i_dst in range(8):
            v = pool[i_dst % 4] ^ hc
            hc = hc * MULT_B
            v = v * hc
            v = v ^ (v >> XSHIFT)
            out[i_dst] = v
        o64 = out.astype(_U64)
        return np.stack([o64[2 * k] | (o64[2 * k + 1] << _U64(32)) for k in range(4)], axis=1)


def _mul64(a, b):
    """full 64x64 -> (hi, lo) on uint64 arrays"""
    a0, a1 = a & _M32, a >> _U64(32)
    b0, b1 = b & _M32, b >> _U64(32)
    p00, p01, p10, p11 = a0 * b0, a0 * b1, a1 * b0, a1 * b1
    mid = (p00 >> _U64(32)) + (p01 & _M32) + (p10 & _M32)
    lo = (p00 & _M32) | (mid << _U64(32))
    hi = p11 + (p01 >> _U64(32)) + (p10 >> _U64(32)) + (mid >> _U64(32))
    return hi, lo


class VecPCG64:
    """n independent PCG64 streams; stream i equals numpy's PCG64(SeedSequence(seeds[i], spawn_key=spawn_key))."""

    def __init__(self, seeds: Optional[np.ndarray] = None, spawn_key: Tuple[int, ...] = ()):
        if seeds is not None:
            self.seed(seeds, spawn_key)

    def seed(self, seeds, spawn_key: Tuple[int, ...] = ()):
        with np.errstate(over="ignore"):
            s = seed_sequence_state(seeds, spawn_key)
            n = len(s)
            init_hi, init_lo, seq_hi, seq_lo = s[:, 0], s[:, 1], s[:, 2], s[:, 3]
            self.inc_hi = (seq_hi << _U64(1)) | (seq_lo >> _U64(63))
            self.inc_lo = (seq_lo << _U64(1)) | _U64(1)
            self.hi, self.lo = np.zeros(n, _U64), np.zeros(n, _U64)
            self._step(np.ones(n, bool))
            lo = self.lo + init_lo
            self.hi = self.hi + init_hi + (lo < self.lo).astype(_U64)
            self.lo = lo
            self._step(np.ones(n, bool))
            self.has32 = np.zeros(n, bool)
            self.buf32 = np.zeros(n, _U32)

    def _step(self, m):
        with np.errstate(over="ignore"):
            hi, lo = self.hi[m], self.lo[m]
            phi, plo = _mul64(lo, PCG_MULT_LO)
            phi = phi + lo * PCG_MULT_HI + hi * PCG_MULT_LO
            nlo = plo + self.inc_lo[m]
            nhi = phi + self.inc_hi[m] + (nlo < plo).astype(_U64)
            self.hi[m], self.lo[m] = nhi, nlo

    def next_uint64(self, m) -> np.ndarray:
        """advance the streams selected by the boolean mask m; returns their outputs (length m.sum())"""
        self._step(m)
        hi, lo = self.hi[m], self.lo[m]
        rot = hi >> _U64(58)
        x = hi ^ lo
        return (x >> rot) | (x << ((_U64(64) - rot) & _U64(63)))

    def next_uint32(self, m) -> np.ndarray:
        """numpy's pcg64_next32: the high half of a 64-bit output is buffered for the next call"""
        out = np.empty(int(m.sum()), _U32)
        idx = np.nonzero(m)[0]
        use_buf = self.has32[idx]
        out[use_buf] = self.buf32[idx[use_buf]]
        self.has32[idx[use_buf]] = False
        fresh = idx[~use_buf]
        if len(fresh):
            fm = np.zeros(len(self.hi), bool)
            fm[fresh] = True
            v = self.next_uint64(fm)
            out[~use_buf] = (v & _M32).astype(_U32)
            self.buf32[fresh] = (v >> _U64(32)).astype(_U32)
            self.has32[fresh] = True
        return out

    def bounded(self, high_excl: int, m: Optional[np.ndarray] = None) -> np.ndarray:
        """Generator.integers(0, high_excl) / the index drawn by Generator.choice(seq of length high_excl), one value per
        selected stream (high_excl <= 2^32): Lemire's method with rejection, on the buffered 32-bit outputs."""
        n = len(self.hi)
        if m is None:
            m = np.ones(n, bool)
        res = np.zeros(n, np.int64)
        rng = int(high_excl) - 1
        if rng == 0:
            return res[m]
        assert 0 < rng <= 0xFFFFFFFF
        rng_excl = _U64(rng + 1)
        threshold = _U64((0xFFFFFFFF - rng) % (rng + 1))
        pending = m.copy()
        first = True
        with np.errstate(over="ignore"):
            while pending.any():
                mm = self.next_uint32(pending).astype(_U64) * rng_excl
                leftover = mm & _M32
                # first round: accept unless leftover < rng_excl and leftover < threshold; later rounds: while leftover < threshold
                reject = (leftover < threshold) & ((leftover < rng_excl) if first else True)
                idx = np.nonzero(pending)[0]
                acc = idx[~reject]
                res[acc] = (mm[~reject] >> _U64(32)).astype(np.int64)
                pending[acc] = False
                first = False
        return res[m]

    # ---- device layout (include/tinycarlo_b200.h TC_RNG_*)
    def device_rows(self) -> np.ndarray:
        buf = np.where(self.has32, (_U64(1) << _U64(32)) | self.buf32.astype(_U64), _U64(0))
        return np.ascontiguousarray(np.stack([self.hi, self.lo, self.inc_hi, self.inc_lo, buf], axis=1).astype(_U64))

    def load_device_rows(self, rows: np.ndarray):
        r = np.asarray(rows).view(_U64).reshape(-1, 5)
        self.hi, self.lo, self.inc_hi, self.inc_lo = (r[:, k].copy() for k in range(4))
        self.has32 = (r[:, 4] >> _U64(32)) != 0
        self.buf32 = (r[:, 4] & _M32).astype(_U32)

    # ---- checkpointing
    def state_dict(self):
        return {k: getattr(self, k).copy() for k in ("hi", "lo", "inc_hi", "inc_lo", "has32", "buf32")}

    def load_state_dict(self, d):
        for k in ("hi", "lo", "inc_hi", "inc_lo", "has32", "buf32"):
            setattr(self, k, np.array(d[k]))
