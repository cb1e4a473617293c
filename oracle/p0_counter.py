"""numpy restatement of the counter-based P_0 of ``tpn_init_projection`` (include/tpnet_b200.h).

For seed s, draw k, node u and column c < d:
    x[0..3] = Philox4x64-10(counter = (c // 4, u, 0, 0), key = (s, k))
    v_i     = ((x_i >> 11) + 0.5) * 2^-53                      (f64, the add rounded to nearest)
    (z_0, z_1), (z_2, z_3) = Box-Muller(v_0, v_1), Box-Muller(v_2, v_3)
                             r = sqrt(-2 log v_even), theta = 6.283185307179586 * v_odd, z = (r cos theta, r sin theta)
    P_0[u, 4 (c // 4) + i] = fl32(z_i * (1 / sqrt(d)))

Philox runs on uint64 arrays, the 128-bit products split into 32-bit halves, so it does not lean on numpy's own
Philox; the CPU suite checks the two agree.  log / sin / cos are numpy's, which are not correctly rounded, nor are the
device's: ``p0_rows`` also returns where the f64 value lies so close to an f32 rounding midpoint that the two may
round apart.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

M0 = np.uint64(0xD2E7470EE14C6C93)
M1 = np.uint64(0xCA5A826395121157)
W0 = np.uint64(0x9E3779B97F4A7C15)
W1 = np.uint64(0xBB67AE8584CAA73B)
_LO32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)

#: f64 ulps around an f32 rounding midpoint inside which device and oracle may round apart
MIDPOINT_ULPS = 64


def mulhilo64(a: np.ndarray, b: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """(high, low) 64-bit words of the 128-bit products a * b of uint64 arrays."""
    a0, a1 = a & _LO32, a >> _S32
    b0, b1 = b & _LO32, b >> _S32
    p00, p01, p10, p11 = a0 * b0, a0 * b1, a1 * b0, a1 * b1
    mid = (p00 >> _S32) + (p01 & _LO32) + (p10 & _LO32)          # < 3 * 2^32: no wrap
    hi = p11 + (p01 >> _S32) + (p10 >> _S32) + (mid >> _S32)
    lo = (mid << _S32) | (p00 & _LO32)
    return hi, lo


def philox4x64_10(ctr: np.ndarray, key: np.ndarray) -> np.ndarray:
    """Philox4x64-10 of counters ``ctr`` [n, 4] under keys ``key`` [n, 2] (or [2]); uint64 in and out."""
    x = [np.array(ctr[:, i], dtype=np.uint64) for i in range(4)]
    key = np.broadcast_to(np.asarray(key, dtype=np.uint64), (len(x[0]), 2))
    k0, k1 = key[:, 0].copy(), key[:, 1].copy()
    with np.errstate(over='ignore'):
        for r in range(10):
            if r:
                k0 += W0
                k1 += W1
            hi0, lo0 = mulhilo64(np.full_like(x[0], M0), x[0])
            hi1, lo1 = mulhilo64(np.full_like(x[2], M1), x[2])
            x = [hi1 ^ x[1] ^ k0, lo1, hi0 ^ x[3] ^ k1, lo0]
    return np.stack(x, axis=1)


def uniform53(x: np.ndarray) -> np.ndarray:
    return ((x >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def normals(seed: int, draw: int, nodes: np.ndarray, dim: int) -> np.ndarray:
    """f64 standard normals z [len(nodes), dim] of columns 0..dim-1 of the given global node ids."""
    nodes = np.asarray(nodes, dtype=np.uint64).reshape(-1)
    blocks = (int(dim) + 3) // 4
    q = np.tile(np.arange(blocks, dtype=np.uint64), len(nodes))
    u = np.repeat(nodes, blocks)
    zero = np.zeros_like(q)
    x = philox4x64_10(np.stack([q, u, zero, zero], axis=1), np.array([seed, draw], dtype=np.uint64))
    v = uniform53(x)
    r01 = np.sqrt(-2.0 * np.log(v[:, 0]))
    r23 = np.sqrt(-2.0 * np.log(v[:, 2]))
    t01 = 6.283185307179586 * v[:, 1]
    t23 = 6.283185307179586 * v[:, 3]
    z = np.stack([r01 * np.cos(t01), r01 * np.sin(t01), r23 * np.cos(t23), r23 * np.sin(t23)], axis=1)
    return z.reshape(len(nodes), blocks * 4)[:, :dim]


def p0_rows(seed: int, draw: int, nodes: np.ndarray, dim: int) -> Tuple[np.ndarray, np.ndarray]:
    """(float32 P_0 rows [len(nodes), dim], bool mask of the entries whose f64 value lies within MIDPOINT_ULPS f64
    ulps of an f32 rounding midpoint — the only entries where another log / sin / cos may round differently)."""
    y = normals(seed, draw, nodes, dim) * (1.0 / np.sqrt(np.float64(dim)))
    f = y.astype(np.float32)
    up = (f.astype(np.float64) + np.nextafter(f, np.float32(np.inf)).astype(np.float64)) / 2
    dn = (f.astype(np.float64) + np.nextafter(f, np.float32(-np.inf)).astype(np.float64)) / 2
    dist = np.minimum(np.abs(y - up), np.abs(y - dn))
    return f, dist <= MIDPOINT_ULPS * np.spacing(np.abs(y))
