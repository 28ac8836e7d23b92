"""Host reference of the counter-based dropout mask defined in csrc/gemm_epilogue.cuh (drop_key / drop_hash2 /
drop_keep): numpy uint32 / uint64 arithmetic that predicts every keep / drop decision of every dropout site bit for bit.

    keep = keep_mask(seed, p, idx, G, epoch)     # bool array shaped like idx

The 64-bit seed (plus epoch * 0xD1B54A32D192ED03, the CUDA-graph replay counter) is mixed by splitmix64 into two 32-bit
keys; one hash of (keys, idx // G) seeds a 32-bit LCG that is stepped (idx % G) + 1 times, and the element is kept iff
the result is >= thr16 << 16 with thr16 = uint32(float32(p) * 65536).

Index spaces of the sites (G = elements per hash):
    GEMM epilogue output   m * N + n                                  G = 8
    act_bwd                flat element index                         G = 8
    layernorm_bwd dx_drop  row * D + col                              G = 8
    attention P            ((b * H + h) * N + q) * ceil16(N) + k      G = 16

The index builders below read the process-wide device epoch counter (src/training/graphs.py) when `epoch` is None, so
a CUDA graph built earlier in the same process does not change what they predict."""
import sys

import numpy as np

M64 = 0xFFFFFFFFFFFFFFFF
EPOCH_MUL = 0xD1B54A32D192ED03
LCG_A, LCG_C = 747796405, 2891336453


def _lcg_tables(G):
    """x_i = seed * mul[i] + add[i] (mod 2^32) after i + 1 LCG steps."""
    mul, add = [], []
    a, c = 1, 0
    for _ in range(G):
        a = (a * LCG_A) & 0xFFFFFFFF
        c = (c * LCG_A + LCG_C) & 0xFFFFFFFF
        mul.append(a)
        add.append(c)
    return np.array(mul, dtype=np.uint32), np.array(add, dtype=np.uint32)


def thr16(p):
    """(uint32)(p * 65536.0f) in float32, as drop_thr16."""
    if p <= 0:
        return 0
    return int(np.float32(p) * np.float32(65536.0))


def inv_keep(p):
    """Rescale of kept elements: 65536 / (65536 - thr16) (1 when p == 0). Equals ops.drop_inv_keep; the kernels hold it
    in float32 (inv_keep_f32)."""
    if p <= 0:
        return 1.0
    return 65536.0 / (65536.0 - thr16(p))


def inv_keep_f32(p):
    return float(np.float32(65536.0) / (np.float32(65536.0) - np.float32(thr16(p)))) if p > 0 else 1.0


def mixed_seed(seed, epoch=0):
    return ((int(seed) & M64) + (int(epoch) & M64) * EPOCH_MUL) & M64


def drop_keys(seed, epoch=0):
    """(s0, s1): splitmix64 of seed + epoch * 0xD1B54A32D192ED03, split into two 32-bit keys."""
    z = (mixed_seed(seed, epoch) + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    z ^= z >> 31
    return z & 0xFFFFFFFF, z >> 32


def hash2(s0, s1, pair):
    """drop_hash2 on a uint64 array of group indices."""
    pair = np.asarray(pair, dtype=np.uint64)
    lo = (pair & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    hi = (pair >> np.uint64(32)).astype(np.uint32)
    x = (lo ^ np.uint32(s0)) * np.uint32(0x9E3779B1)
    x ^= x >> np.uint32(15)
    x = (x + hi * np.uint32(0x632BE5AB) + np.uint32(s1)) * np.uint32(0x85EBCA77)
    x ^= x >> np.uint32(13)
    x *= np.uint32(0xC2B2AE3D)
    x ^= x >> np.uint32(16)
    return x


def keep_mask(seed, p, idx, G, epoch=0):
    """Keep decisions (bool, shaped like idx) of the elements with flat dropout indices `idx` (uint64-convertible)."""
    idx = np.asarray(idx, dtype=np.uint64)
    if p <= 0:
        return np.ones(idx.shape, dtype=bool)
    s0, s1 = drop_keys(seed, epoch)
    mul, add = _lcg_tables(G)
    h = hash2(s0, s1, idx // np.uint64(G))
    pos = (idx % np.uint64(G)).astype(np.intp)
    x = h * mul[pos] + add[pos]
    return x >= np.uint32(thr16(p) << 16)


def current_epoch():
    """Value of the process-wide dropout epoch counter (0 when no CUDA graph has registered one)."""
    graphs = sys.modules.get("src.training.graphs")
    if graphs is None or not graphs._epoch:
        return 0
    (t,) = graphs._epoch.values()
    return int(t.item())


def _epoch(epoch):
    return current_epoch() if epoch is None else epoch


def ceil16(n):
    return (n + 15) & ~15


def attn_index(B, H, N, Nk=None):
    """[B, H, N, N] attention dropout indices ((b * H + h) * N + q) * ceil16(N) + k (keys limited to Nk when given)."""
    Nk = N if Nk is None else Nk
    bh = np.arange(B * H, dtype=np.uint64).reshape(B, H, 1, 1)
    q = np.arange(N, dtype=np.uint64).reshape(1, 1, N, 1)
    k = np.arange(Nk, dtype=np.uint64).reshape(1, 1, 1, Nk)
    return (bh * np.uint64(N) + q) * np.uint64(ceil16(N)) + k


def attn_mask(B, H, N, seed, p, epoch=None):
    """[B, H, N(query), N(key)] keep mask of the attention probabilities."""
    epoch = _epoch(epoch)
    out = np.empty((B, H, N, N), dtype=bool)
    idx = attn_index(1, 1, N)[0, 0]
    for bh in range(B * H):               # one (image, head) at a time: bounded temporaries at N = 4096
        out[bh // H, bh % H] = keep_mask(seed, p, idx + np.uint64(bh * N * ceil16(N)), 16, epoch)
    return out


def gemm_mask(M, N, seed, p, epoch=None):
    """[M, N] keep mask of a GEMM epilogue output (also layernorm_bwd's dx_drop with N = D)."""
    idx = np.arange(M, dtype=np.uint64)[:, None] * np.uint64(N) + np.arange(N, dtype=np.uint64)[None, :]
    return keep_mask(seed, p, idx, 8, _epoch(epoch))


ln_mask = gemm_mask


def flat_mask(n, seed, p, epoch=None):
    """[n] keep mask of act_bwd (flat element index)."""
    return keep_mask(seed, p, np.arange(n, dtype=np.uint64), 8, _epoch(epoch))
