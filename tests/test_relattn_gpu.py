"""GPU: relative-position attention core (forward + backward) against the oracle's closed form.  With attention dropout
on, the reference applies the very mask the kernels generate, regenerated on the host (dropmask.py)."""
import math

import pytest
import torch

import dropmask as D
import txl_oracle as O
from attn_readout import attn_readout, shifted

pytestmark = pytest.mark.gpu
HS = 64
SEED, SITE = 2 ** 40 + 12345, 2 ** 33 + 9  # above 2^32: both halves of the 64-bit hash inputs take part


@pytest.fixture(autouse=True)
def _no_step_counter():
    """The host masks below assume no step counter; an earlier test may have registered the process-wide one."""
    with D.pinned_step_counter(None):
        yield


def _ref(q, k, v, r, u, vb, reset, B, N, Q, M, dh, mem_len, same_length, keep=None):
    """fp64 autograd reference built from the oracle pieces.  q [Q,B,N,dh], k/v [K,B,N,dh], r [K,N,dh].
    keep: fp64 [B,N,Q,K] dropout factor (mask / (1 - p)) on the probabilities; lse is the logsumexp before dropout."""
    K = M + Q
    mask = O.attn_mask(Q, M, mem_len, same_length, reset, B)
    ac = torch.einsum("ibnd,jbnd->bnij", q + u, k)
    bd = O.rel_shift_gather(torch.einsum("ibnd,jnd->bnij", q + vb, r), Q)
    s = (ac + bd) / math.sqrt(dh)
    s = s.masked_fill(mask[:, None], float("-inf"))
    p = torch.softmax(s, -1)
    if keep is not None:
        p = p * keep
    return torch.einsum("bnij,jbnd->ibnd", p, v), torch.logsumexp(s, -1)


def _msl(Q, M, mem_len, same_length):
    ml = M + Q - mem_len
    return Q - ml if same_length and ml > 0 else Q


def _pad_heads(x, dtype):  # [..., N, dh] -> [..., N*64]
    out = torch.zeros(*x.shape[:-1], HS, dtype=torch.float32)
    out[..., : x.shape[-1]] = x
    return out.reshape(*x.shape[:-2], -1).to("cuda").to(dtype).contiguous()


CASES = [  # B, N, Q, M, dh, mem_len, same_length, reset
    (2, 3, 5, 0, 10, 8, False, False),
    (3, 2, 8, 16, 10, 16, False, True),
    (2, 2, 8, 12, 50, 12, True, True),
    (2, 10, 16, 24, 50, 24, False, True),
    (4, 2, 1, 37, 50, 64, False, False),      # decode shape
    (1, 2, 128, 128, 50, 128, False, False),  # one full tile
    (2, 2, 128, 256, 50, 256, True, True),
    (2, 1, 64, 200, 50, 200, False, False),
]
# + drop_p, K / V base 16- but not 32-byte aligned
FWD_BWD_CASES = [c + (0.0, False) for c in CASES] + [c + (0.1, False) for c in CASES] + [
    (3, 5, 1, 130, 50, 130, False, True, 0.1, False),    # Q = 1: B * N and K not multiples of 4
    (2, 20, 1, 200, 50, 128, True, False, 0.1, False),   # Q = 1, N > 16 heads: 4-warp CTAs; first kept key 73
    (4, 3, 1, 0, 50, 8, False, False, 0.1, False),       # Q = 1 without memory
    (3, 5, 1, 130, 50, 130, False, True, 0.1, True),     # Q = 1, K / V 16-byte aligned: the generic kernels
    (2, 3, 33, 40, 50, 73, False, True, 0.1, False),     # partial tcgen05 tiles
    (2, 2, 100, 60, 50, 60, True, True, 0.1, False),
    (2, 2, 200, 96, 50, 128, True, True, 0.1, False),    # tcgen05 forward over two query tiles, SIMT backward
    (2, 10, 128, 1024, 50, 1024, False, True, 0.1, False),  # the benchmarked MLE shape
    (2, 2, 64, 64, 50, 64, False, True, 0.5, False),
]


@pytest.mark.parametrize("impl", [1, 0])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", FWD_BWD_CASES)
def test_relattn_fwd_bwd(case, dtype, impl):
    """Every forward kernel (single-token, decode, SIMT, tcgen05) and every backward path (fused single-token, SIMT
    with the small-Q or the per-key pass, tcgen05), with and without dropout, against fp64 autograd."""
    from tgan_b200 import lib as L
    B, N, Q, M, dh, mem_len, same_length, use_reset, drop_p, unaligned = case
    if dtype == torch.float32 and impl == 0:
        pytest.skip("fp32 always runs the SIMT kernels")
    K = M + Q
    g = torch.Generator().manual_seed(B * 1000 + Q * 10 + M)
    rnd = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    q, k, v, r = rnd(Q, B, N, dh), rnd(K, B, N, dh), rnd(K, B, N, dh), rnd(K, N, dh)
    u, vb = 0.3 * rnd(N, dh), 0.3 * rnd(N, dh)
    do = rnd(Q, B, N, dh)
    reset = torch.zeros(B, dtype=torch.bool)
    if use_reset and M > 0:
        reset[B - 1] = True
    # round inputs to the compute dtype first so the reference sees the same operands
    rd = lambda t: t.to(dtype).double()
    q, k, v, r, do = rd(q), rd(k), rd(v), rd(r), rd(do)
    keep = D.as_scale(D.attn_keep(SEED, SITE, B, N, Q, K, drop_p), drop_p) if drop_p > 0 else None
    leaves = [t.requires_grad_(True) for t in (q, k, v, r, u, vb)]
    out_ref, lse_ref = _ref(q, k, v, r, u, vb, reset, B, N, Q, M, dh, mem_len, same_length, keep)
    (out_ref * do).sum().backward()

    qd, dod = _pad_heads(q.detach().reshape(Q * B, N, dh), dtype), _pad_heads(do.reshape(Q * B, N, dh), dtype)
    kvd = torch.cat([_pad_heads(k.detach().reshape(K * B, N, dh), dtype),
                     _pad_heads(v.detach().reshape(K * B, N, dh), dtype)], 1).contiguous()
    rdv = _pad_heads(r.detach(), dtype)
    ud, vbd = _pad_heads(u.detach(), torch.float32).view(-1), _pad_heads(vb.detach(), torch.float32).view(-1)
    NH = N * HS
    off = 16 // kvd.element_size() if unaligned else 0
    kvin = shifted(kvd, off) if unaligned else kvd
    out = torch.empty(Q * B, NH, device="cuda", dtype=dtype)
    lse = torch.empty(B * N * Q, device="cuda")
    rs = reset.to(torch.uint8).cuda() if use_reset else None
    msl = _msl(Q, M, mem_len, same_length)
    scale = 1 / math.sqrt(dh)
    L.relattn_fwd(qd, kvin, kvin, 2 * NH, rdv, ud, vbd, rs, out, lse, B, N, Q, M, msl, same_length, scale, drop_p, SEED,
                  SITE, impl=impl, k_off=off, v_off=off + NH)
    torch.cuda.synchronize()
    tol = 2e-5 if dtype == torch.float32 else 2e-2
    got = out.float().cpu().view(Q, B, N, HS)
    assert (got[..., :dh].double() - out_ref.detach()).abs().max() < tol
    assert torch.all(got[..., dh:] == 0)
    # the tensor-core path rounds (q + u), (q + v) to bf16 operands: ~0.4% of the score magnitude
    assert (lse.cpu().view(B, N, Q).double() - lse_ref.detach()).abs().max() < (1e-4 if dtype == torch.float32 else 2e-2)

    dq = torch.empty_like(qd)
    dkv = torch.empty_like(kvd)
    dr = torch.empty(K, NH, device="cuda")
    du, dvb = torch.zeros(NH, device="cuda"), torch.zeros(NH, device="cuda")
    delta = torch.empty(B * N * max(Q, M + 1 if Q == 1 else Q), device="cuda")
    L.relattn_bwd(qd, kvin, kvin, 2 * NH, rdv, ud, vbd, rs, out, dod, lse, delta, dq, dkv, dkv, 2 * NH, dr, du, dvb,
                  B, N, Q, M, msl, same_length, scale, drop_p, SEED, SITE, impl=impl, k_off=off, v_off=off + NH,
                  dv_off=NH)
    torch.cuda.synchronize()
    gt = 2e-4 if dtype == torch.float32 else 6e-2

    def chk(name, got, want):
        want = want.double()
        err = (got.double().cpu() - want).abs().max().item()
        assert err <= gt * max(1.0, want.abs().max().item()), (name, err, want.abs().max().item())

    chk("dq", dq.float().view(Q, B, N, HS)[..., :dh], leaves[0].grad)
    chk("dk", dkv[:, :NH].float().reshape(K, B, N, HS)[..., :dh], leaves[1].grad)
    chk("dv", dkv[:, NH:].float().reshape(K, B, N, HS)[..., :dh], leaves[2].grad)
    chk("dr", dr.view(K, N, HS)[..., :dh], leaves[3].grad)
    chk("du", du.view(N, HS)[:, :dh], leaves[4].grad)
    chk("dvb", dvb.view(N, HS)[:, :dh], leaves[5].grad)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("Q,M,impl,unaligned", [(1, 40, 1, False),   # relattn_dec_fwd
                                                (1, 40, 1, True),    # relattn_fwd_simt at Q = 1
                                                (4, 40, 1, False),   # relattn_fwd_decode
                                                (16, 30, 1, False),  # relattn_fwd_simt
                                                (48, 16, 2, False)])  # relattn_fwd_tc_kernel
def test_relattn_dropout_mask_readout(Q, M, impl, unaligned, dtype):
    if impl == 2 and dtype == torch.float32:
        pytest.skip("the tcgen05 kernel is bf16 only")
    attn_readout(Q, M, dtype, impl, unaligned, 0.25, SEED, SITE)


SPLIT_CASES = [  # B, N, M, mem_len, same_length, reset, dtype, drop_p
    (4, 2, 37, 64, False, False, torch.bfloat16, 0.0),
    (3, 5, 130, 130, False, True, torch.float32, 0.1),
    (37, 10, 133, 128, True, True, torch.bfloat16, 0.1),  # B > 32: second block row of the memory-side kernel
    (2, 20, 1, 1, False, False, torch.float32, 0.1),
    (5, 3, 0, 8, False, False, torch.bfloat16, 0.1),      # memory side without memory rows
]


@pytest.mark.parametrize("case", SPLIT_CASES)
def test_relattn_bwd_step_split_matches_fused_and_reference(case):
    """tgan_relattn_bwd_step: phase 1 (query side) then phase 2 (memory side) after a single-token forward.  Phase 1
    writes dq and the dk / dv of key row M only (the engine points dk / dv at a shifted base, so any other row would land
    outside its buffer) and leaves du / dvb alone; phase 2 writes the rows j < M, all of dR and adds to du / dvb."""
    from tgan_b200 import lib as L
    B, N, M, mem_len, same_length, use_reset, dtype, drop_p = case
    Q, K, dh, NH = 1, M + 1, 50, N * HS
    g = torch.Generator().manual_seed(B * 100 + M)
    rnd = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    rd = lambda t: t.to(dtype).double()
    q, k, v, r, do = rd(rnd(Q, B, N, dh)), rd(rnd(K, B, N, dh)), rd(rnd(K, B, N, dh)), rd(rnd(K, N, dh)), rd(rnd(Q, B, N, dh))
    u, vb = 0.3 * rnd(N, dh), 0.3 * rnd(N, dh)
    reset = torch.zeros(B, dtype=torch.bool)
    if use_reset and M > 0:
        reset[0] = reset[B - 1] = True
    keep = D.as_scale(D.attn_keep(SEED, SITE, B, N, Q, K, drop_p), drop_p) if drop_p > 0 else None
    leaves = [t.requires_grad_(True) for t in (q, k, v, r, u, vb)]
    out_ref, _ = _ref(q, k, v, r, u, vb, reset, B, N, Q, M, dh, mem_len, same_length, keep)
    (out_ref * do).sum().backward()

    qd, dod = _pad_heads(q.detach().reshape(B, N, dh), dtype), _pad_heads(do.reshape(B, N, dh), dtype)
    kv = torch.cat([_pad_heads(k.detach().reshape(K * B, N, dh), dtype),
                    _pad_heads(v.detach().reshape(K * B, N, dh), dtype)], 1).contiguous()
    rdv = _pad_heads(r.detach(), dtype)
    ud, vbd = _pad_heads(u.detach(), torch.float32).view(-1), _pad_heads(vb.detach(), torch.float32).view(-1)
    rs = reset.to(torch.uint8).cuda() if use_reset else None
    msl, scale = _msl(Q, M, mem_len, same_length), 1 / math.sqrt(dh)
    out, lse = torch.empty(B, NH, device="cuda", dtype=dtype), torch.empty(B * N, device="cuda")
    L.relattn_fwd(qd, kv, kv, 2 * NH, rdv, ud, vbd, rs, out, lse, B, N, Q, M, msl, same_length, scale, drop_p, SEED, SITE,
                  v_off=NH)
    args = (B, N, M, msl, same_length, scale, drop_p, SEED, SITE)

    # fused single-token backward
    dq_f, dkv_f = torch.empty_like(qd), torch.empty_like(kv)
    dr_f, du_f, dvb_f = torch.empty(K, NH, device="cuda"), torch.zeros(NH, device="cuda"), torch.zeros(NH, device="cuda")
    delta = torch.empty(B * N * K, device="cuda")
    L.relattn_bwd(qd, kv, kv, 2 * NH, rdv, ud, vbd, rs, out, dod, lse, delta, dq_f, dkv_f, dkv_f, 2 * NH, dr_f, du_f,
                  dvb_f, B, N, Q, M, msl, same_length, scale, drop_p, SEED, SITE, v_off=NH, dv_off=NH)

    # split backward on sentinel-filled outputs
    SENT = -77.0
    dq, dkv, dr = torch.full_like(qd, SENT), torch.full_like(kv, SENT), torch.full((K, NH), SENT, device="cuda")
    du0, dvb0 = torch.linspace(-1, 1, NH, device="cuda"), torch.linspace(2, -2, NH, device="cuda")
    du, dvb = du0.clone(), dvb0.clone()
    scratch = torch.empty(2 * B * N * K + 2 * B * N * HS, device="cuda")
    L.relattn_bwd_step(1, qd, kv, kv, 2 * NH, rdv, ud, vbd, rs, out, dod, lse, scratch, dq, dkv, dkv, 2 * NH, dr, du, dvb,
                       *args, v_off=NH, dv_off=NH)
    torch.cuda.synchronize()
    rows = dkv.view(K, B, 2 * NH)
    assert torch.equal(dq, dq_f), "phase 1 dq differs from the fused backward"
    assert torch.equal(rows[M], dkv_f.view(K, B, 2 * NH)[M]), "phase 1 dk / dv of key row M differ from the fused backward"
    assert torch.all(rows[:M] == SENT), "phase 1 wrote a memory row of dk / dv"
    assert torch.all(dr == SENT), "phase 1 wrote dR"
    assert torch.equal(du, du0) and torch.equal(dvb, dvb0), "phase 1 changed du / dvb"
    row_m = rows[M].clone()
    L.relattn_bwd_step(2, qd, kv, kv, 2 * NH, rdv, ud, vbd, rs, out, dod, lse, scratch, dq, dkv, dkv, 2 * NH, dr, du, dvb,
                       *args, v_off=NH, dv_off=NH)
    torch.cuda.synchronize()
    assert torch.equal(dkv, dkv_f), "split dk / dv differ from the fused backward"
    assert torch.equal(rows[M], row_m), "phase 2 rewrote key row M"
    assert torch.equal(dq, dq_f)
    assert torch.all(dr.view(K, N, HS)[..., dh:] == 0), "dR pad lanes not zero"

    def chk(name, got, want, tol):
        want = want.double()
        err = (got.double().cpu() - want).abs().max().item()
        assert err <= tol * max(1.0, want.abs().max().item()), (name, err, want.abs().max().item())

    gt = 2e-4 if dtype == torch.float32 else 6e-2
    chk("dq", dq.float().view(B, N, HS)[..., :dh], leaves[0].grad[0], gt)
    chk("dk", dkv[:, :NH].float().reshape(K, B, N, HS)[..., :dh], leaves[1].grad, gt)
    chk("dv", dkv[:, NH:].float().reshape(K, B, N, HS)[..., :dh], leaves[2].grad, gt)
    chk("dr", dr.view(K, N, HS)[..., :dh], leaves[3].grad, gt)
    chk("du", (du - du0).view(N, HS)[:, :dh], leaves[4].grad, gt)
    chk("dvb", (dvb - dvb0).view(N, HS)[:, :dh], leaves[5].grad, gt)
    # atomics in another order: the fused path's fp32 reductions agree to rounding
    chk("dr fused", dr_f, dr.cpu(), 1e-5)
    chk("du fused", du_f, (du - du0).cpu(), 1e-5)
    chk("dvb fused", dvb_f, (dvb - dvb0).cpu(), 1e-5)


@pytest.mark.parametrize("case", [(2, 2, 128, 256, 256, False, True), (3, 1, 64, 100, 128, True, False),
                                  (2, 3, 128, 1024, 1024, False, False)])
def test_relattn_tcgen05_matches_simt_with_dropout(case):
    """bf16: the tcgen05 kernels (forced) against the SIMT kernels on identical inputs, attention dropout ON --
    both generate the mask from the same counter hash, so outputs and every gradient must agree."""
    from tgan_b200 import lib as L
    B, N, Q, M, mem_len, same_length, use_reset = case
    dh, K, NH = 50, M + Q, N * HS
    g = torch.Generator().manual_seed(Q + M)
    mk = lambda rows: _pad_heads(torch.randn(rows, N, dh, generator=g), torch.bfloat16)
    q, kk, vv, r, do = mk(Q * B), mk(K * B), mk(K * B), mk(K), mk(Q * B)
    kv = torch.cat([kk, vv], 1).contiguous()
    u = _pad_heads(0.3 * torch.randn(N, dh, generator=g), torch.float32).view(-1)
    vb = _pad_heads(0.3 * torch.randn(N, dh, generator=g), torch.float32).view(-1)
    rs = None
    if use_reset:
        rs = torch.zeros(B, dtype=torch.uint8)
        rs[0] = 1
        rs = rs.cuda()
    msl = Q
    if same_length:
        ml = K - mem_len
        msl = Q - ml if ml > 0 else Q
    scale = 1 / math.sqrt(dh)
    res = {}
    for impl in (1, 2):
        out = torch.empty(Q * B, NH, device="cuda", dtype=torch.bfloat16)
        lse = torch.empty(B * N * Q, device="cuda")
        L.relattn_fwd(q, kv, kv, 2 * NH, r, u, vb, rs, out, lse, B, N, Q, M, msl, same_length, scale, 0.1, 7, 3,
                      impl=impl, v_off=NH)
        dq, dkv = torch.empty_like(q), torch.full_like(kv, 7.0)
        dr = torch.full((K, NH), 7.0, device="cuda")
        du, dvb = torch.zeros(NH, device="cuda"), torch.zeros(NH, device="cuda")
        delta = torch.empty(B * N * max(Q, M + 1 if Q == 1 else Q), device="cuda")
        # both backward passes consume the SAME forward result so only the backward kernels differ
        o_in, l_in = (out, lse) if impl == 1 else (res[1][0], res[1][1])
        L.relattn_bwd(q, kv, kv, 2 * NH, r, u, vb, rs, o_in, do, l_in, delta, dq, dkv, dkv, 2 * NH, dr, du, dvb, B, N,
                      Q, M, msl, same_length, scale, 0.1, 7, 3, impl=impl, v_off=NH, dv_off=NH)
        torch.cuda.synchronize()
        res[impl] = (out, lse, dq.float(), dkv.float(), dr, du, dvb)
    names = ["out", "lse", "dq", "dkv", "dr", "du", "dvb"]
    for nm, a, b in zip(names, res[1], res[2]):
        a, b = a.float(), b.float()
        tol = 3e-2 * max(1.0, a.abs().max().item())
        assert (a - b).abs().max().item() < tol, (nm, (a - b).abs().max().item(), a.abs().max().item())
        rel = (a - b).norm().item() / max(a.norm().item(), 1e-6)
        assert rel < 2e-2, (nm, rel)


def test_relattn_tcgen05_lazy_rescale_large_dynamic_range():
    """Scores whose running maximum keeps growing along the keys (by far more than 2^8 per tile) force the
    forward's lazy rescale of the TMEM-resident output on many tiles; compare with the SIMT kernel."""
    from tgan_b200 import lib as L
    B, N, Q, M, dh = 2, 2, 128, 384, 50
    K, NH = M + Q, N * HS
    g = torch.Generator().manual_seed(5)
    qf = torch.randn(Q * B, N, dh, generator=g)
    kf = torch.randn(K, B, N, dh, generator=g) * torch.linspace(0.1, 12.0, K).view(K, 1, 1, 1)
    vf = torch.randn(K * B, N, dh, generator=g)
    q, kk, vv = _pad_heads(qf, torch.bfloat16), _pad_heads(kf.reshape(K * B, N, dh), torch.bfloat16), _pad_heads(vf, torch.bfloat16)
    r = _pad_heads(torch.randn(K, N, dh, generator=g), torch.bfloat16)
    kv = torch.cat([kk, vv], 1).contiguous()
    u, vb = torch.zeros(NH, device="cuda"), torch.zeros(NH, device="cuda")
    res = {}
    for impl in (1, 2):
        out = torch.empty(Q * B, NH, device="cuda", dtype=torch.bfloat16)
        lse = torch.empty(B * N * Q, device="cuda")
        L.relattn_fwd(q, kv, kv, 2 * NH, r, u, vb, None, out, lse, B, N, Q, M, Q, False, 1 / math.sqrt(dh), 0.0, 0, 0,
                      impl=impl, v_off=NH)
        torch.cuda.synchronize()
        res[impl] = (out.float(), lse)
    assert torch.isfinite(res[2][0]).all() and torch.isfinite(res[2][1]).all()
    assert (res[1][0] - res[2][0]).abs().max().item() < 3e-2 * max(1.0, res[1][0].abs().max().item())
    assert (res[1][1] - res[2][1]).abs().max().item() < 2e-2 * max(1.0, res[1][1].abs().max().item())
