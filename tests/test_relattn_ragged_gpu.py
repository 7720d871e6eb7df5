"""GPU: the attention forward with a per-sequence key floor (tgan_relattn_fwd_ragged: left-padded prompts of different
lengths) against an fp64 reference, on every forward kernel, and bit-identical to tgan_relattn_fwd when the floor is
off."""
import math

import pytest
import torch

import txl_oracle as O
from test_relattn_gpu import CASES, HS, _pad_heads

pytestmark = pytest.mark.gpu


def _ref(q, k, v, r, u, vb, reset, floors, B, N, Q, M, dh, mem_len, same_length):
    """test_relattn_gpu._ref plus the floor: key j of row i of sequence b is masked iff j < min(floors[b], i + M).
    floors[b] = max(reset[b] ? M : 0, key_start[b] - key_base), clamped to [0, K]."""
    K = M + Q
    mask = O.attn_mask(Q, M, mem_len, same_length, reset, B)
    i = torch.arange(Q).view(1, Q, 1)
    j = torch.arange(K).view(1, 1, K)
    mask = mask | (j < torch.minimum(floors.view(B, 1, 1), i + M))
    ac = torch.einsum("ibnd,jbnd->bnij", q + u, k)
    bd = O.rel_shift_gather(torch.einsum("ibnd,jnd->bnij", q + vb, r), Q)
    s = (ac + bd) / math.sqrt(dh)
    s = s.masked_fill(mask[:, None], float("-inf"))
    p = torch.softmax(s, -1)
    return torch.einsum("bnij,jbnd->ibnd", p, v), torch.logsumexp(s, -1)


def _inputs(B, N, Q, M, dh, dtype, seed):
    K = M + Q
    g = torch.Generator().manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    rd = lambda t: t.to(dtype).double()  # the reference sees the operands the kernel sees
    q, k, v, r = rd(rnd(Q, B, N, dh)), rd(rnd(K, B, N, dh)), rd(rnd(K, B, N, dh)), rd(rnd(K, N, dh))
    u, vb = 0.3 * rnd(N, dh), 0.3 * rnd(N, dh)
    dev = dict(q=_pad_heads(q.reshape(Q * B, N, dh), dtype),
               kv=torch.cat([_pad_heads(k.reshape(K * B, N, dh), dtype),
                             _pad_heads(v.reshape(K * B, N, dh), dtype)], 1).contiguous(),
               r=_pad_heads(r, dtype), u=_pad_heads(u, torch.float32).view(-1), vb=_pad_heads(vb, torch.float32).view(-1))
    return (q, k, v, r, u, vb), dev


def _msl(Q, M, mem_len, same_length):
    if not same_length:
        return Q
    ml = M + Q - mem_len
    return Q - ml if ml > 0 else Q


# offsets key_start[b] - key_base per sequence: 0, inside a 32-key tile, on a tile boundary, beyond the first rows' own
# positions (pad query rows), below key_base (a window that has slid past the pads), and the floor of a fully padded
# memory that ends exactly at the first query row
def _offsets(Q, M):
    return [0, 13, 64, M + Q // 2 + 1, -7, M]


# B is the number of offsets; reset marks sequences 1 and 4 (under, resp. instead of, the floor)
RAGGED_CASES = [  # N, Q, M, dh, mem_len, same_length, use_reset, dtype, impl
    (2, 1, 70, 50, 70, False, False, torch.float32, 0),     # Q = 1: relattn_dec_fwd
    (2, 1, 70, 50, 70, True, True, torch.bfloat16, 0),
    (3, 6, 40, 50, 40, False, True, torch.float32, 0),      # Q <= 8: relattn_fwd_decode
    (2, 5, 80, 50, 80, True, False, torch.bfloat16, 1),
    (2, 20, 50, 50, 50, False, True, torch.float32, 0),     # 8 < Q < 32: relattn_fwd_simt
    (2, 20, 60, 50, 60, True, False, torch.bfloat16, 1),
    (2, 128, 200, 50, 200, False, True, torch.bfloat16, 2),  # Q >= 32, bf16: relattn_fwd_tc_kernel
    (2, 200, 96, 50, 160, True, True, torch.bfloat16, 2),   # two query tiles, the second partial, same_length
    (1, 64, 0, 50, 64, False, False, torch.bfloat16, 2),    # context pass of a fresh ring: no memory at all
]


@pytest.mark.parametrize("case", RAGGED_CASES)
def test_relattn_fwd_ragged_matches_reference(case):
    from tgan_b200 import lib as L
    N, Q, M, dh, mem_len, same_length, use_reset, dtype, impl = case
    K = M + Q
    offs = _offsets(Q, M)
    B = len(offs)
    (q, k, v, r, u, vb), d = _inputs(B, N, Q, M, dh, dtype, seed=Q * 7 + M)
    reset = torch.zeros(B, dtype=torch.bool)
    if use_reset and M > 0:
        reset[1] = reset[4] = True
    key_base = 1000
    key_start = torch.tensor([key_base + o for o in offs], dtype=torch.int32)
    floors = torch.tensor(offs).clamp(0, K)
    floors = torch.where(reset, torch.maximum(floors, torch.tensor(M)), floors)
    out_ref, lse_ref = _ref(q, k, v, r, u, vb, reset, floors, B, N, Q, M, dh, mem_len, same_length)

    NH = N * HS
    out = torch.empty(Q * B, NH, device="cuda", dtype=dtype)
    lse = torch.empty(B * N * Q, device="cuda")
    L.relattn_fwd(d["q"], d["kv"], d["kv"], 2 * NH, d["r"], d["u"], d["vb"],
                  reset.to(torch.uint8).cuda() if use_reset else None, out, lse, B, N, Q, M,
                  _msl(Q, M, mem_len, same_length), same_length, 1 / math.sqrt(dh), 0.0, 0, 0, impl=impl, v_off=NH,
                  key_start=key_start.cuda(), key_base=key_base)
    torch.cuda.synchronize()
    got = out.float().cpu().view(Q, B, N, HS)
    assert torch.isfinite(got).all() and torch.isfinite(lse).all()
    tol = 2e-5 if dtype == torch.float32 else 2e-2
    assert (got[..., :dh].double() - out_ref).abs().max() < tol
    assert torch.all(got[..., dh:] == 0)
    assert (lse.cpu().view(B, N, Q).double() - lse_ref).abs().max() < (1e-4 if dtype == torch.float32 else 2e-2)
    # a pad query row (i + M below its sequence's floor) attends to itself only: its output is its own v row
    n_pad = 0
    for b in range(B):
        for i in range(Q):
            if i + M < floors[b]:
                assert (got[i, b, :, :dh].double() - v[i + M, b]).abs().max() < tol, (b, i)
                n_pad += 1
    assert n_pad > 0


@pytest.mark.parametrize("impl", [1, 0])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", CASES)
def test_relattn_fwd_ragged_without_floor_is_bit_identical(case, dtype, impl):
    """key_start all equal to key_base puts every floor at 0 (or at M for a reset row): the same arithmetic as
    tgan_relattn_fwd, bit for bit."""
    from tgan_b200 import lib as L
    B, N, Q, M, dh, mem_len, same_length, use_reset = case
    if dtype == torch.float32 and impl == 0:
        pytest.skip("fp32 always runs the SIMT kernels")
    _, d = _inputs(B, N, Q, M, dh, dtype, seed=B * 1000 + Q * 10 + M)
    rs = None
    if use_reset and M > 0:
        rs = torch.zeros(B, dtype=torch.uint8)
        rs[B - 1] = 1
        rs = rs.cuda()
    NH = N * HS
    res = []
    for key_start in (None, torch.full((B,), 4242, dtype=torch.int32, device="cuda")):
        out = torch.full((Q * B, NH), 3.0, device="cuda", dtype=dtype)
        lse = torch.full((B * N * Q,), 3.0, device="cuda")
        L.relattn_fwd(d["q"], d["kv"], d["kv"], 2 * NH, d["r"], d["u"], d["vb"], rs, out, lse, B, N, Q, M,
                      _msl(Q, M, mem_len, same_length), same_length, 1 / math.sqrt(dh), 0.0, 0, 0, impl=impl, v_off=NH,
                      key_start=key_start, key_base=4242)
        res.append((out, lse))
    torch.cuda.synchronize()
    assert torch.equal(res[0][0], res[1][0])
    assert torch.equal(res[0][1], res[1][1])


def test_relattn_fwd_ragged_rejects_a_bad_key_start():
    from tgan_b200 import lib as L
    B, N, Q, M = 2, 1, 4, 8
    _, d = _inputs(B, N, Q, M, 50, torch.float32, seed=1)
    out, lse = torch.empty(Q * B, HS, device="cuda"), torch.empty(B * N * Q, device="cuda")
    for bad in (torch.zeros(B, dtype=torch.int64, device="cuda"), torch.zeros(B + 1, dtype=torch.int32, device="cuda")):
        with pytest.raises(L.TganError):
            L.relattn_fwd(d["q"], d["kv"], d["kv"], 2 * HS, d["r"], d["u"], d["vb"], None, out, lse, B, N, Q, M, Q,
                          False, 0.1, 0.0, 0, 0, v_off=HS, key_start=bad, key_base=0)
