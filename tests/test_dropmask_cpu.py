"""CPU: the host port of the dropout mask hash (tests/dropmask.py) against the __host__ functions of common.cuh.

A small harness includes the header, evaluates every mask helper on a fixed table of inputs and prints the results;
the port must reproduce them bit for bit.  This fails as soon as the hash in common.cuh changes without the port."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import dropmask as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "transformer-gan_b200", "csrc", "common.cuh")

HARNESS = r"""
#include "%s"
#include <stdlib.h>
void tgan_set_error(const char*, ...) {}
int main(int argc, char** argv) {
    FILE* f = fopen(argv[1], "r");
    unsigned long long seed, site, e, row, j;
    char ps[64];
    while (fscanf(f, "%%llu %%llu %%llu %%llu %%llu %%63s", &seed, &site, &e, &row, &j, ps) == 6) {
        const uint32_t th = dropout_thresh16(strtof(ps, nullptr));
        const uint32_t key = dropout_key(seed, site);
        const uint32_t rk = attn_drop_rowkey(key, (uint32_t)row);
        printf("%%u %%u %%u %%u %%d %%u %%u %%u %%d %%u %%u\n", mix32((uint32_t)seed), key, th,
               dropout_hash_pair(key, e >> 1), (int)dropout_keep_k(key, e, th), dropout_keep8_k(key, e, th), rk,
               attn_drop_pair(rk, (uint32_t)j >> 1), (int)attn_drop_keep(rk, (int)j, th), attn_mixlite((uint32_t)row),
               dropout_thresh(strtof(ps, nullptr)));
    }
    fclose(f);
    return 0;
}
"""

PROBS = ["1e-5", "0.1", "0.25", "0.5", "0.9"]


def _inputs(n=1000):
    rng = np.random.default_rng(2024)
    u64 = lambda: rng.integers(0, 2 ** 64, n, dtype=np.uint64)
    seed, site = u64(), u64()
    seed[:8] = [0, 1, 7, 42, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 5, 2 ** 64 - 1]
    site[:8] = [0, 3, 17, 2 ** 32 + 1, 2 ** 40, 5, 2 ** 63, 2 ** 64 - 1]
    # element indices: small, odd and even, and above 2^32 (pair index crosses 2^31 / 2^32)
    e = rng.integers(0, 2 ** 40, n, dtype=np.uint64)
    e[: n // 4] = rng.integers(0, 4096, n // 4, dtype=np.uint64)
    e[n // 4: n // 4 + 6] = [2 ** 32 - 2, 2 ** 32 - 1, 2 ** 32, 2 ** 32 + 1, 2 ** 33 + 1, 2 ** 63 + 3]
    # row ids near the uint32 wrap, keys 0 .. 2^20
    row = rng.integers(0, 2 ** 32, n, dtype=np.uint64)
    row[:6] = [0, 1, 2 ** 31, 2 ** 32 - 2, 2 ** 32 - 1, 12345]
    j = rng.integers(0, 2 ** 20, n, dtype=np.uint64)
    j[:4] = [0, 1, 2 ** 20 - 2, 2 ** 20 - 1]
    ps = [PROBS[i % len(PROBS)] for i in range(n)]
    return seed, site, e, row, j, ps


def _port(seed, site, e, row, j, ps):
    out = np.zeros((len(seed), 11), dtype=np.uint64)
    for p in PROBS:
        sel = np.array([x == p for x in ps])
        th = D.thresh16(float(p))
        key = D.dropout_key(seed[sel], site[sel])
        rk = D.attn_drop_rowkey(key, row[sel])
        e8 = e[sel][:, None] + np.arange(8, dtype=np.uint64)[None, :]
        keep8 = (D.dropout_keep_k(key[:, None], e8, th).astype(np.uint64) << np.arange(8, dtype=np.uint64)).sum(1)
        out[sel] = np.stack([D.mix32(seed[sel]), key, np.full(sel.sum(), th, np.uint64),
                             D.dropout_hash_pair(key, e[sel] >> np.uint64(1)), D.dropout_keep_k(key, e[sel], th),
                             keep8, rk, D.attn_drop_pair(rk, j[sel] >> np.uint64(1)), D.attn_drop_keep(rk, j[sel], th),
                             D.attn_mixlite(row[sel]), np.full(sel.sum(), th, np.uint64)], 1).astype(np.uint64)
    return out


def test_thresholds():
    assert D.thresh16(0.1) == 6554 and D.thresh16(0.25) == 16384 and D.thresh16(0.0) == 0 and D.thresh16(1.0) == 65535


def test_port_matches_common_cuh_bit_for_bit(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    src = tmp_path / "harness.cu"
    src.write_text(HARNESS % HEADER)
    exe = tmp_path / "harness"
    cc = subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(exe), str(src)],
                        capture_output=True, text=True)
    assert cc.returncode == 0, f"the harness including common.cuh does not compile:\n{cc.stderr}"
    seed, site, e, row, j, ps = _inputs()
    table = tmp_path / "inputs.txt"
    table.write_text("".join(f"{a} {b} {c} {d} {x} {p}\n" for a, b, c, d, x, p in zip(seed, site, e, row, j, ps)))
    res = subprocess.run([str(exe), str(table)], check=True, capture_output=True, text=True).stdout.split("\n")
    got = np.array([[int(x) for x in line.split()] for line in res if line], dtype=np.uint64)
    want = _port(seed, site, e, row, j, ps)
    assert got.shape == want.shape
    bad = np.argwhere(got != want)
    assert bad.size == 0, [(int(r), int(c), int(got[r, c]), int(want[r, c])) for r, c in bad[:10]]
    # the keep bits are not degenerate: every threshold drops roughly p of the elements
    for p in PROBS:
        sel = np.array([x == p for x in ps])
        assert abs(1 - got[sel, 4].mean() - float(p)) < 0.1
