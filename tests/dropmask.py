"""Host port of the dropout mask generator in transformer-gan_b200/csrc/common.cuh.

Every dropout mask of the library is a stateless integer hash of (seed, site, element index), so the host can
regenerate it bit for bit.  The functions below mirror the __host__ __device__ helpers of common.cuh one to one,
vectorised over numpy uint64 arrays and masked to 32 bits after every multiply.  tests/test_dropmask_cpu.py checks
them against the header itself; the GPU tests use the mask builders to compare dropout-on kernels with fp64
references that apply the very same mask.
"""
import contextlib

import numpy as np
import torch

M32 = np.uint64(0xFFFFFFFF)


def _u64(x):
    return np.asarray(x, dtype=np.uint64)


def _mul(a, c):
    return (_u64(a) * np.uint64(c)) & M32


def mix32(x):
    x = _u64(x) & M32
    x ^= x >> np.uint64(16)
    x = _mul(x, 0x7FEB352D)
    x ^= x >> np.uint64(15)
    x = _mul(x, 0x846CA68B)
    x ^= x >> np.uint64(16)
    return x


def dropout_key(seed, site):
    seed, site = _u64(seed), _u64(site)
    lo, hi = np.uint64(32), M32
    inner = mix32(((site >> lo) + np.uint64(0x9E3779B9)) & hi)
    return mix32((seed & hi) ^ mix32((seed >> lo) ^ mix32((site & hi) ^ inner)))


def step_fold(key, counter):
    """common.cuh step_fold with the registered device counter holding `counter` (None: no counter)."""
    if counter is None:
        return _u64(key)
    return mix32(_u64(key) ^ _mul(counter, 0x9E3779B1))


def dropout_hash_pair(key, pair):
    pair = _u64(pair)
    return mix32(_mul(pair & M32, 0x9E3779B1) ^ _mul(pair >> np.uint64(32), 0x85EBCA77) ^ _u64(key))


def _half(h, odd, thresh):
    return np.where(odd, h >> np.uint64(16), h & np.uint64(0xFFFF)) >= np.uint64(thresh)


def dropout_keep_k(key, e, thresh):
    e = _u64(e)
    return _half(dropout_hash_pair(key, e >> np.uint64(1)), (e & np.uint64(1)) != 0, thresh)


def attn_drop_rowkey(key, row):
    return mix32(_u64(key) ^ _mul(_u64(row) & M32, 0x9E3779B1))


def attn_mixlite(x):
    p = (_u64(x) & M32) * np.uint64(0x9E3779B1)
    return _mul((p >> np.uint64(32)) ^ (p & M32), 0x7FEB352D)


def attn_drop_pair(rowkey, j_pair):
    return attn_mixlite((_u64(rowkey) + _mul(j_pair, 0x85EBCA77)) & M32)


def attn_drop_keep(rowkey, j, thresh):
    j = _u64(j)
    return _half(attn_drop_pair(rowkey, j >> np.uint64(1)), (j & np.uint64(1)) != 0, thresh)


def thresh16(p):
    """dropout_thresh16: p is a C float, widened to double before the rounding."""
    t = float(np.float32(p)) * 65536.0 + 0.5
    return int(min(max(t, 0.0), 65535.0))


# ---- mask builders, in the index convention of the kernels (bool numpy arrays, True = kept) ------------------
def elem_keep(seed, site, rows, cols, ld, p, step=None):
    """Element masks (GEMM epilogue, tgan_dropout, embed_fwd / embed_bwd, ln_bwd, pos_emb): index row * ld + col."""
    key = step_fold(dropout_key(seed, site), step)
    e = np.arange(rows, dtype=np.uint64)[:, None] * np.uint64(ld) + np.arange(cols, dtype=np.uint64)[None, :]
    return dropout_keep_k(key, e, thresh16(p))


def attn_keep(seed, site, B, N, Q, K, p, step=None):
    """Relative-attention probability mask [B, N, Q, K]: row id (b * N + n) * Q + i as uint32, key j."""
    key = step_fold(dropout_key(seed, site), step)
    rows = np.arange(B * N * Q, dtype=np.uint64) & M32
    rk = attn_drop_rowkey(key, rows)[:, None]
    return attn_drop_keep(rk, np.arange(K, dtype=np.uint64)[None, :], thresh16(p)).reshape(B, N, Q, K)


def bert_keep(seed, site, B, heads, T, p, step=None):
    """BERT attention probability mask [B, heads, T, T]: element ((b * heads + h) * T + i) * T + j."""
    key = step_fold(dropout_key(seed, site), step)
    e = np.arange(B * heads * T * T, dtype=np.uint64)
    return dropout_keep_k(key, e, thresh16(p)).reshape(B, heads, T, T)


def as_scale(keep, p):
    """fp64 tensor keep / (1 - p): the factor the kernels apply to a kept element (1 everywhere when p == 0)."""
    keep = torch.from_numpy(np.ascontiguousarray(keep))
    return keep.double() / (1.0 - p) if p > 0 else torch.ones(keep.shape, dtype=torch.float64)


@contextlib.contextmanager
def pinned_step_counter(value, device="cuda"):
    """Register a device step counter holding `value` (None: no counter) for the duration of the block, so that the
    host masks can fold in the same value.  On exit the process-wide counter of the device, if one exists, is
    registered again; otherwise none is."""
    from tgan_b200 import lib
    ctr = None
    if value is not None:
        ctr = torch.tensor([value], dtype=torch.int32, device=device)
    lib.set_step_counter(ctr)
    try:
        yield ctr
    finally:
        torch.cuda.synchronize()
        lib.set_step_counter(lib._step_counters.get(torch.device(device).index or 0))
