"""numpy restatement of the library's Philox4x32-10 generator and of the three dropout masks built on it.  TEST INFRASTRUCTURE ONLY.

Follows end-to-end-slu_b200/csrc/philox.cuh: the 64-bit counter is (c0 = low word, c1 = high word, c2 = c3 = 0), the key is the
64-bit seed (k0 = low word, k1 = high word), bumped by (0x9E3779B9, 0xBB67AE85) after each of the 10 rounds.  The masks:
  dropout_mask       slu_dropout_mask: counter = index i of the float4 group, word k -> element 4i+k, keep: word < keep_threshold(p)
  gru_mask           slu_dropout_mask_gru and the GRU kernels: element (b, t, col) of [B][T][256], counter
                     ((b*256 + col) << 32) | (t >> 3), 16-bit draw t & 7 (bits 16*(k&1) of word k>>1), keep: draw < keep_threshold16(p)
  cell_mask          csrc/decoder.cu cell_mask: element e of a [B][D] cell output at decoder step `step`, counter (step << 40) | (e >> 2),
                     word e & 3, keep: word < keep_threshold(p), key seed ^ seed_word when the kernels are given a device seed word
Kept elements carry float32(1 / (1 - p)) with p as the float32 the C ABI receives, computed in double.
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def philox4x32_10(ctr, seed):
    """ctr: array of 64-bit counters, seed: 64-bit key -> uint32 array [4, *ctr.shape] (the four output words)."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    zero = np.zeros_like(ctr)
    return philox4x32_10_words((ctr & _LO, ctr >> _32, zero, zero), int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF)


def philox4x32_10_words(c, k0, k1):
    """The generator on a full 128-bit counter (c0, c1, c2, c3 arrays of 32-bit values) and key (k0, k1): Random123's definition,
    of which the library uses the c2 = c3 = 0 half."""
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) for x in c)
    for _ in range(10):
        p0, p1 = c0 * _M0, c2 * _M1                      # 32 x 32 -> 64-bit products: exact in uint64
        c0, c1, c2, c3 = (p1 >> _32) ^ c1 ^ np.uint64(k0), p1 & _LO, (p0 >> _32) ^ c3 ^ np.uint64(k1), p0 & _LO
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3]).astype(np.uint32)


def _p32(p):
    return float(np.float32(p))


def keep_threshold(p):
    """slu_keep_threshold: P(keep) = threshold / 2^32 for 32-bit draws."""
    th = (1.0 - _p32(p)) * 4294967296.0
    return 0xFFFFFFFF if th >= 4294967295.0 else int(th)


def keep_threshold16(p):
    """slu_keep_threshold16: P(keep) = threshold / 2^16 for 16-bit draws, rounded; never 0 (0 means "no dropout")."""
    th = (1.0 - _p32(p)) * 65536.0 + 0.5
    t = 65536 if th >= 65536.0 else int(th)
    return 1 if t == 0 else t


def keep_scale(p):
    return np.float32(1.0 / (1.0 - _p32(p)))


def dropout_mask(n, p, seed):
    """slu_dropout_mask: float32 [n] of {0, 1/(1-p)}."""
    w = philox4x32_10(np.arange((n + 3) // 4, dtype=np.uint64), seed)          # [4, groups]
    keep = w.T.reshape(-1)[:n] < np.uint32(keep_threshold(p))
    return np.where(keep, keep_scale(p), np.float32(0)).astype(np.float32)


def gru_mask(B, T, p, seed):
    """slu_dropout_mask_gru: float32 [B][T][256] of {0, 1/(1-p)}."""
    b = np.arange(B, dtype=np.uint64)[:, None, None]
    t = np.arange(T, dtype=np.uint64)[None, :, None]
    col = np.arange(256, dtype=np.uint64)[None, None, :]
    w = philox4x32_10(((b * np.uint64(256) + col) << _32) | (t >> np.uint64(3)), seed)        # [4, B, T, 256]
    k = (t & np.uint64(7)).astype(np.int64)
    word = np.take_along_axis(w, np.broadcast_to(k >> 1, (1, B, T, 256)), 0)[0]
    draw = (word >> (16 * (k & 1)).astype(np.uint32)) & np.uint32(0xFFFF)
    return np.where(draw < keep_threshold16(p), keep_scale(p), np.float32(0)).astype(np.float32)


def cell_mask(B, D, p, seed, step, seed_word=None):
    """The decoder's inter-cell Dropout at step `step` (slu_grucell_fwd / _bwd): float32 [B][D] of {0, 1/(1-p)}; all ones at p = 0."""
    if _p32(p) == 0.0:
        return np.ones((B, D), np.float32)
    key = int(seed) ^ (0 if seed_word is None else int(seed_word))
    e = np.arange(B * D, dtype=np.uint64)
    w = philox4x32_10((np.uint64(step) << np.uint64(40)) | (e >> np.uint64(2)), key)            # [4, B*D]
    word = w[(e & np.uint64(3)).astype(np.int64), np.arange(B * D)]
    return np.where(word < np.uint32(keep_threshold(p)), keep_scale(p), np.float32(0)).astype(np.float32).reshape(B, D)
