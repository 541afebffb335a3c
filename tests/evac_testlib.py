"""Shared helpers for the parity tests (test infrastructure)."""
from __future__ import annotations

import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.evac_oracle import OracleConfig, OracleEnv, compute_statuses  # noqa: F401

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN_DIR = os.path.join(HERE, "golden")


def golden_names():
    return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith(".npz"))


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    case = json.loads(str(z["case_json"]))
    return case, z


def oracle_config_from_case(case) -> OracleConfig:
    kw = dict(case["env"])
    kw.update(case["wrap"])
    return OracleConfig(**kw)


def case_noise(case):
    """Dense noise table [T,N] of an 'injected' golden case (same construction as
    tests/golden/gen_golden.py::case_inputs)."""
    T = case["steps"]
    n = case["env"].get("number_of_pedestrians", 10)
    c = case["env"].get("noise_coef", 0.2)
    noise = np.random.RandomState(5000 + case["seed"]).uniform(-c / 2, c / 2, size=(T, n))
    return noise.astype(np.float32).astype(np.float64)


def make_oracle_at_golden_start(case, z) -> OracleEnv:
    """Oracle env whose state equals the reference's state right after reset()."""
    env = OracleEnv(oracle_config_from_case(case))
    env.set_state(z["init_positions"], z["init_directions"], z["init_statuses"], np.zeros(2, np.float32))
    env.n_episodes = 1
    return env


# ---------------------------------------------------------------------------------------------
# NumPy restatement of the library's counter-based random streams (csrc/philox.cuh) so the
# in-kernel RNG can be fed to the oracle bit for bit.
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
STREAM_NOISE, STREAM_RESET, STREAM_AGENT = 0, 1, 2


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10; inputs broadcastable uint32 arrays; returns 4 uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & 0xFFFFFFFF for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0 & 0xFFFFFFFF), np.uint64(k1 & 0xFFFFFFFF)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(_M0) * c[0]
        p1 = np.uint64(_M1) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(_W0)) & mask
        k1 = (k1 + np.uint64(_W1)) & mask
    return [x.astype(np.uint32) for x in c]


def evac_random(seed, stream, env, episode, now, ped):
    k0 = (seed & 0xFFFFFFFF) ^ ((stream * _W0) & 0xFFFFFFFF)
    k1 = (seed >> 32) & 0xFFFFFFFF
    return philox4x32_10(ped, now, episode, env, k0, k1)


def u01(r):
    return (np.asarray(r, dtype=np.uint32) >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)


_M2 = 0xD256D193


def philox2x32_10(c0, c1, k):
    """Vectorised Philox2x32-10 (csrc/philox.cuh::philox2x32_10); returns 2 uint32 arrays."""
    c0, c1, k = (np.asarray(x, dtype=np.uint64) & np.uint64(0xFFFFFFFF) for x in np.broadcast_arrays(c0, c1, k))
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p = np.uint64(_M2) * c0
        hi, lo = p >> np.uint64(32), p & mask
        c0, c1 = hi ^ k ^ c1, lo
        k = (k + np.uint64(_W0)) & mask
    return c0.astype(np.uint32), c1.astype(np.uint32)


def evac_key32(seed, stream, episode):
    return ((seed & 0xFFFFFFFF) ^ ((((seed >> 32) & 0xFFFFFFFF) * _W0) & 0xFFFFFFFF) ^ ((episode * _W1) & 0xFFFFFFFF)
            ^ ((stream * 0x85EBCA6B) & 0xFFFFFFFF))


def philox_noise(seed, env, episode, now, n, noise_coef):
    """Dense [n] float32 noise the kernels draw for (env, episode, step-in-episode `now`): pedestrian i reads word
    (i >> 5) & 1 of Philox2x32 block (i & 31) | (i >> 6) << 5, counter ((block & 2047) | now << 11, env), the upper block
    bits (pedestrians >= 4096) folded into the key."""
    i = np.arange(n, dtype=np.int64)
    block = (i & 31) | ((i >> 6) << 5)
    key = np.uint64(evac_key32(seed, STREAM_NOISE, episode)) ^ ((block >> 11).astype(np.uint64) * np.uint64(0xC2B2AE35) & np.uint64(0xFFFFFFFF))
    r = philox2x32_10((block & 2047) | (now << 11), env, key)
    words = np.where(((i >> 5) & 1) == 1, r[1], r[0])
    return (u01(words) - np.float32(0.5)) * np.float32(noise_coef)


def philox_action(seed, env, episode, now):
    r = philox2x32_10(now << 11, env, evac_key32(seed, STREAM_AGENT, episode))
    return np.array([np.float32(2) * u01(r[0]) - np.float32(1), np.float32(2) * u01(r[1]) - np.float32(1)], dtype=np.float32).reshape(2)


# ---------------------------------------------------------------------------------------------
# NumPy restatement of the fused policy's two streams (csrc/evac_policy.cuh): the dropout masks of the embedding kernel in
# training mode and the Normal draws of the heads.  Seeds and stream offsets are 64-bit, env_g is the global env index
# (env_index_offset + e, taken mod 2^32).
_U32 = np.uint64(0xFFFFFFFF)
PW_MAX_S = 64


def _u32(x):
    return np.asarray(x, dtype=np.uint64) & _U32


def fmix32(h):
    h = _u32(h)
    h = h ^ (h >> np.uint64(16))
    h = (h * np.uint64(0x85EBCA6B)) & _U32
    h = h ^ (h >> np.uint64(13))
    h = (h * np.uint64(0xC2B2AE35)) & _U32
    return h ^ (h >> np.uint64(16))


def drop_base_key(seed, offset, env_g):
    seed_lo, seed_hi, off_lo, off_hi = (np.uint64(v) for v in (seed & 0xFFFFFFFF, seed >> 32, offset & 0xFFFFFFFF, offset >> 32))
    inner = fmix32((_u32(env_g) * np.uint64(0x9E3779B1) + off_lo) & _U32)
    return fmix32(seed_lo ^ inner ^ ((seed_hi * np.uint64(0x85EBCA77)) & _U32) ^ ((off_hi * np.uint64(0xC2B2AE3D)) & _U32))


def drop_row_key(base, blk, row):
    return fmix32(_u32(base) ^ ((_u32(np.asarray(blk) * PW_MAX_S + np.asarray(row)) * np.uint64(0x27D4EB2F)) & _U32))


def drop_word(row_key, k):
    """16-bit word k of a row's stream: k = c is the attention output's feature c, k = 8 + c the block output's."""
    k = _u32(k)
    t = fmix32(_u32(row_key) + (k >> np.uint64(1)) * np.uint64(0x9E3779B9))
    return np.where((k & np.uint64(1)) == 1, t >> np.uint64(16), t & np.uint64(0xFFFF))


def drop_ff_word(row_key, g):
    return fmix32(_u32(row_key) + (np.uint64(8) + _u32(g)) * np.uint64(0x9E3779B9))


def drop_ff_mix(t):
    t = (_u32(t) * np.uint64(0x9E3779B1)) & _U32
    return t ^ (t >> np.uint64(15))


def drop_hidden_words(row_key, F):
    """16-bit words of hidden features 0 .. F - 1: feature 4g + 2i + j is half j of word i of group g, word 0 = drop_ff_word,
    word 1 = drop_ff_mix of it."""
    f = np.arange(F, dtype=np.uint64)
    w = drop_ff_word(np.asarray(row_key)[..., None], f >> np.uint64(2))
    w = np.where(((f >> np.uint64(1)) & np.uint64(1)) == 1, drop_ff_mix(w), w)
    return np.where((f & np.uint64(1)) == 1, w >> np.uint64(16), w & np.uint64(0xFFFF))


def drop_site_words(seed, offset, env_g, blk, row, D, F):
    """The 16-bit words of the three dropout sites of block `blk`, row `row` (broadcastable): attention output [.., D],
    feed-forward hidden layer [.., F], block output [.., D]."""
    key = drop_row_key(drop_base_key(seed, offset, env_g), blk, row)[..., None]
    c = np.arange(D)
    return drop_word(key, c), drop_hidden_words(key[..., 0], F), drop_word(key, 8 + c)


def drop_threshold(p):
    """lrint(p * 65536) of the float32 dropout probability: a word below it drops its element."""
    return int(np.rint(np.float64(np.float32(p)) * 65536.0))


def dropout_masks(seed, offset, env_index_offset, E, num_blocks, S, D, F, p):
    """Per block, the float32 masks (attention [E, S, D], hidden [E, S, F], output [E, S, D]) of one forward call with stream
    offset `offset`: 0 where dropped, float32(1 / (1 - p)) where kept."""
    thr = np.uint64(drop_threshold(p))
    keep = np.float32(1) / (np.float32(1) - np.float32(p))
    env_g = (env_index_offset + np.arange(E, dtype=np.int64)) & 0xFFFFFFFF
    rows = np.arange(S)
    out = []
    for b in range(num_blocks):
        words = drop_site_words(seed, offset, env_g[:, None], b, rows[None, :], D, F)
        out.append(tuple(np.where(w < thr, np.float32(0), keep).astype(np.float32) for w in words))
    return out


def policy_normal(seed, offset, env_g, A):
    """[.., A] standard Normal draws of the heads: Philox4x32-10 counter (env_g, offset lo, offset hi, 'POLI'), key = seed;
    24-bit uniforms u = ((w >> 8) + 0.5) * 2^-24 and the angle 2 pi u formed in float32 as the kernel forms them, Box-Muller
    in float64: words (0, 1) give components 0 (cos) and 1 (sin), words (2, 3) component 2 (cos).  Returns (z, radius)."""
    r = philox4x32_10(_u32(env_g), offset & 0xFFFFFFFF, offset >> 32, 0x504F4C49, seed & 0xFFFFFFFF, seed >> 32)
    u = [((w >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24) for w in r]
    rad = [np.sqrt(-2.0 * np.log(u[p].astype(np.float64))) for p in (0, 2)]
    ang = [(np.float32(2 * np.pi) * u[p]).astype(np.float64) for p in (1, 3)]
    z = np.stack([rad[0] * np.cos(ang[0]), rad[0] * np.sin(ang[0]), rad[1] * np.cos(ang[1])], axis=-1)
    return z[..., :A], np.stack([rad[0], rad[0], rad[1]], axis=-1)[..., :A]


def philox_layout(seed, env, episode, n, dtype=np.float32):
    """(positions [n,2], directions [n,2]) of a kernel-side reset (csrc/evac_kernels.cuh::random_layout)."""
    r = evac_random(seed, STREAM_RESET, env, episode, 0, np.arange(n))
    two, one = np.float32(2), np.float32(1)
    px, py, vx, vy = (two * u01(r[i]) - one for i in range(4))
    pos = np.stack([px, py], axis=1).astype(dtype)
    v = np.stack([vx, vy], axis=1).astype(dtype)
    v[(v[:, 0] == 0) & (v[:, 1] == 0), 0] = 1
    nrm = np.sqrt(v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1])
    return pos, (v / nrm[:, None]).astype(dtype)
