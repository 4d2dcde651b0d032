"""numpy reference of the package's dropout mask (DESIGN.md section 3.16), for tests only: Philox4x32-10 and the keep rule.

Element e of a call's contiguous [rows, C] output draws
    u(e) = (r[(e & 7) >> 1] >> (16 * (e & 1))) & 0xFFFF,
    r = Philox4x32-10(counter (lo32(e >> 3), hi32(e >> 3), 0, 0), key (lo32(key), hi32(key)))
and is kept iff u(e) >= t, t = floor(p * 65536 + 0.5) with p as the float32 the C ABI takes; kept values are scaled by
float32(1 / (1 - p)).
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr uint32 [..., 4], key uint32 [..., 2] (broadcast) -> uint32 [..., 4]."""
    c = [np.asarray(ctr[..., i], dtype=np.uint32) for i in range(4)]
    k0 = np.asarray(key[..., 0], dtype=np.uint32)
    k1 = np.asarray(key[..., 1], dtype=np.uint32)
    with np.errstate(over="ignore"):
        for r in range(10):
            if r:
                k0 = k0 + _W0
                k1 = k1 + _W1
            p0 = _M0 * c[0].astype(np.uint64)
            p1 = _M1 * c[2].astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), (p0 & _LO).astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), (p1 & _LO).astype(np.uint32)
            c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, -1)


def rule(p):
    """(t, scale) of the keep rule at rate p (p in (0, 1))."""
    p32 = np.float32(p)
    return int(np.floor(np.float64(p32) * 65536.0 + 0.5)), float(np.float32(1.0 / (1.0 - np.float64(p32))))


def draws(key, n):
    """16-bit draws u(e) of elements 0 .. n-1 under the int64 key."""
    k = int(key) & 0xFFFFFFFFFFFFFFFF
    groups = np.arange((n + 7) // 8, dtype=np.uint64)
    ctr = np.zeros(groups.shape + (4,), dtype=np.uint32)
    ctr[:, 0] = (groups & _LO).astype(np.uint32)
    ctr[:, 1] = (groups >> np.uint64(32)).astype(np.uint32)
    r = philox4x32_10(ctr, np.array([k & 0xFFFFFFFF, k >> 32], dtype=np.uint32))       # [groups, 4]
    u = np.stack([r & 0xFFFF, r >> 16], -1).reshape(-1)                                   # element order 0..7 per group
    return u[:n].astype(np.uint32)


def keep_mask(key, n, p):
    """bool [n]: element kept."""
    return draws(key, n) >= rule(p)[0]
