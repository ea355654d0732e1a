"""ORACLE (test infrastructure only): numpy restatement of the sensing and actuation of the ground-plant loop (include/wbc.h,
wbc_loop; csrc/wbc_loop.cuh), written from its definition:

    draw j in [0, 18) of step c:  Philox4x32-10, counter (j, stream, c_lo, c_hi), key (seed_lo, seed_hi) -> w0..w3
    u_a = (((w1 << 32) | w0) >> 11) 2^-53 + 2^-54,  u_b the same of (w3, w2)
    z[2j] = sqrt(-2 ln u_a) cos(2 pi u_b),  z[2j+1] = sqrt(-2 ln u_a) sin(2 pi u_b)
    observe: q_obs quaternion = normalize(dq (x) q), dq the rotation by sigma_rot z[0:3]; every other block value + sigma z
             (z[3:6] base position, z[6:18] joints, z[18:21] angular, z[21:24] linear, z[24:36] joint velocities); sigma = 0
             copies the block
    actuate: hist[c mod 16] = tau_c; applied = strength hist[max(c - d, 0) mod 16]; tick = c + 1
    bad profile (delay outside [0, 15], a sigma or the strength negative or not finite, tick < 0): observed without noise,
             applied 0, status WBC_ST_BADLOOP, hist and tick unchanged

Philox4x32-10 is the generator of Salmon, Moraes, Dror and Shaw, "Parallel random numbers: as easy as 1, 2, 3" (SC 2011), the
function cuRAND calls curand_Philox4x32_10."""
from __future__ import annotations

import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
DRAWS = 18
HIST = 16
ST_BADLOOP = 4096
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr [..., 4], key [..., 2] (uint32) -> [..., 4] uint32; ten rounds, the key bumped between rounds."""
    c = [np.asarray(ctr, np.uint64)[..., k] & _MASK for k in range(4)]
    k0, k1 = (np.asarray(key, np.uint64)[..., k] & _MASK for k in range(2))
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c[0], np.uint64(M1) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & _MASK, p1 >> np.uint64(32), p1 & _MASK
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0, k1 = (k0 + np.uint64(W0)) & _MASK, (k1 + np.uint64(W1)) & _MASK
    return np.stack(c, axis=-1).astype(np.uint32)


def uniforms(w):
    """w [..., 4] -> (u_a, u_b), both in (0, 1)."""
    w = np.asarray(w, np.uint64)
    a = ((w[..., 1] << np.uint64(32)) | w[..., 0]) >> np.uint64(11)
    b = ((w[..., 3] << np.uint64(32)) | w[..., 2]) >> np.uint64(11)
    return a.astype(np.float64) * 2.0**-53 + 2.0**-54, b.astype(np.float64) * 2.0**-53 + 2.0**-54


def normals(seed, stream, c):
    """The 36 normals of step(s) c of stream(s) `stream` under `seed` -> [..., 36] (stream and c broadcast)."""
    stream, c = np.broadcast_arrays(np.asarray(stream, np.int64) & 0xFFFFFFFF, np.asarray(c, np.int64))
    j = np.arange(DRAWS, dtype=np.uint64)
    shape = stream.shape + (DRAWS,)
    cu = c.astype(np.uint64)
    ctr = np.stack([np.broadcast_to(j, shape), np.broadcast_to(stream.astype(np.uint64)[..., None], shape),
                    np.broadcast_to((cu & _MASK)[..., None], shape), np.broadcast_to((cu >> np.uint64(32))[..., None], shape)], axis=-1)
    s = np.uint64(int(seed) & 0xFFFFFFFFFFFFFFFF)
    key = np.broadcast_to(np.array([s & _MASK, s >> np.uint64(32)], np.uint64), shape + (2,))
    ua, ub = uniforms(philox4x32_10(ctr, key))
    r = np.sqrt(-2.0 * np.log(ua))
    z = np.empty(shape + (2,))
    z[..., 0], z[..., 1] = r * np.cos(np.pi * (2.0 * ub)), r * np.sin(np.pi * (2.0 * ub))
    return z.reshape(stream.shape + (2 * DRAWS,))


def profile_ok(noise, delay, strength, tick):
    """Per robot: delay in [0, 15], every sigma and the strength finite and >= 0, tick >= 0."""
    noise = np.asarray(noise, float).reshape(-1, 6)
    return ((np.asarray(delay) >= 0) & (np.asarray(delay) < HIST) & np.isfinite(strength) & (np.asarray(strength) >= 0)
            & np.isfinite(noise).all(axis=1) & (noise >= 0).all(axis=1) & (np.asarray(tick) >= 0))


def quat_mul(a, b):
    """Hamilton product a (x) b of [w x y z] quaternions."""
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    return np.array([aw * bw - ax * bx - ay * by - az * bz, aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx, aw * bz + ax * by - ay * bx + az * bw])


def observe(q, v, sigma, z):
    """One robot: true q [19], v [18], sigma [6], normals z [36] -> q_obs, v_obs."""
    q, v = np.asarray(q, float), np.asarray(v, float)
    qo, vo = q.copy(), v.copy()
    if sigma[0] != 0.0:
        d = sigma[0] * z[0:3]
        th = np.sqrt(d @ d)
        dq = np.array([1.0, 0.0, 0.0, 0.0]) if th == 0.0 else np.concatenate([[np.cos(th / 2)], np.sin(th / 2) * d / th])
        p = quat_mul(dq, q[0:4])
        qo[0:4] = p / np.sqrt(p @ p)
    for blk, (dst, lo, hi, zlo) in enumerate([(qo, 4, 7, 3), (qo, 7, 19, 6)], start=1):
        if sigma[blk] != 0.0:
            dst[lo:hi] = dst[lo:hi] + sigma[blk] * z[zlo:zlo + hi - lo]
    for blk, (lo, hi, zlo) in enumerate([(0, 3, 18), (3, 6, 21), (6, 18, 24)], start=3):
        if sigma[blk] != 0.0:
            vo[lo:hi] = vo[lo:hi] + sigma[blk] * z[zlo:zlo + hi - lo]
    return qo, vo


def observe_batch(q, v, noise, seed, stream, tick, ok=None):
    """N robots: noise [N][6] (sigma), stream [N], tick [N]; a robot with ok[i] False is observed without noise."""
    q, v = np.asarray(q, float), np.asarray(v, float)
    n = len(q)
    noise = np.broadcast_to(np.asarray(noise, float), (n, 6))
    z = normals(seed, stream, np.maximum(np.asarray(tick), 0))
    qo, vo = np.empty_like(q), np.empty_like(v)
    for i in range(n):
        sg = noise[i] if ok is None or ok[i] else np.zeros(6)
        qo[i], vo[i] = observe(q[i], v[i], sg, z[i])
    return qo, vo


class Actuator:
    """The delay ring and motor strength of one robot: command(tau) returns the applied torque of this step."""

    def __init__(self, delay=0, strength=1.0, hist=None, tick=0):
        self.d, self.s = int(delay), float(strength)
        self.hist = np.zeros((HIST, 12)) if hist is None else np.array(hist, float)
        self.tick = int(tick)

    def command(self, tau):
        c = self.tick
        self.hist[c % HIST] = tau
        out = self.s * self.hist[max(c - self.d, 0) % HIST]
        self.tick = c + 1
        return out
