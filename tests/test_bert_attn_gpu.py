"""GPU: the BERT discriminator's attention tiles (tgan_bert_attn_fwd / _bwd / _jvp) against fp64 autograd, with and
without attention dropout.  The reference applies the kernels' own mask, regenerated on the host (dropmask.py).

bf16 with d_head a multiple of 16 runs the mma.sync kernels (bert_attn_mma.cu); fp32, and bf16 with any other d_head
(multiple of 8), run the SIMT kernels (bert_ops.cu)."""
import math

import pytest
import torch

import dropmask as D

pytestmark = pytest.mark.gpu
SEED, SITE = 2 ** 36 + 77, 2 ** 34 + 3
SENT = -55.0
B, HEADS = 3, 12

IMPLS = [(torch.bfloat16, 16), (torch.bfloat16, 32), (torch.bfloat16, 64),                          # mma
         (torch.float32, 8), (torch.float32, 24), (torch.float32, 64),                              # SIMT fp32
         (torch.bfloat16, 8), (torch.bfloat16, 24), (torch.bfloat16, 40), (torch.bfloat16, 56)]     # SIMT bf16


@pytest.fixture(autouse=True)
def _no_step_counter():
    """The host masks below assume no step counter; an earlier test may have registered the process-wide one."""
    with D.pinned_step_counter(None):
        yield


def _ref(qkv, T, dh, keep):
    """qkv fp64 [B*T, 3H] = [Q | K | V], head h at columns h*dh of each third -> ctx [B*T, H], lse [B*heads*T]"""
    x = qkv.view(B, T, 3, HEADS, dh).permute(2, 0, 3, 1, 4)  # [3, B, heads, T, dh]
    s = x[0] @ x[1].transpose(-1, -2) / math.sqrt(dh)
    p = torch.softmax(s, -1) * keep
    ctx = (p @ x[2]).permute(0, 2, 1, 3).reshape(B * T, HEADS * dh)
    return ctx, torch.logsumexp(s, -1).reshape(-1)


@pytest.mark.parametrize("drop_p", [0.0, 0.1])
@pytest.mark.parametrize("T", [1, 7, 16, 33, 63, 64])
@pytest.mark.parametrize("dtype,dh", IMPLS)
def test_bert_attn_fwd_bwd_jvp(dtype, dh, T, drop_p):
    from tgan_b200 import lib as L
    H = HEADS * dh
    pad = 16 if T % 2 else 0  # odd T: row pitches wider than 3H / H, whose extra columns must stay untouched
    g = torch.Generator().manual_seed(dh * 100 + T)
    rnd = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64).to(dtype).double()
    qkv, dctx, qkvd = rnd(B * T, 3 * H), rnd(B * T, H), rnd(B * T, 3 * H)
    keep = D.as_scale(D.bert_keep(SEED, SITE, B, HEADS, T, drop_p), drop_p)

    def dev(x, cols):
        t = torch.full((B * T, cols + pad), SENT, device="cuda", dtype=dtype)
        t[:, :cols] = x.to(dtype).cuda()
        return t

    qkv_d, dctx_d, qkvd_d = dev(qkv, 3 * H), dev(dctx, H), dev(qkvd, 3 * H)
    ctx = torch.full((B * T, H + pad), SENT, device="cuda", dtype=dtype)
    ctxd = torch.full_like(ctx, SENT)
    dqkv = torch.full((B * T, 3 * H + pad), SENT, device="cuda", dtype=dtype)
    lse = torch.full((B * HEADS * T,), SENT, device="cuda")
    L.bert_attn_fwd(qkv_d, ctx, lse, B, HEADS, T, dh, drop_p, SEED, SITE)
    L.bert_attn_bwd(qkv_d, dctx_d, lse, dqkv, B, HEADS, T, dh, drop_p, SEED, SITE)
    L.bert_attn_jvp(qkv_d, qkvd_d, lse, ctxd, B, HEADS, T, dh, drop_p, SEED, SITE)
    torch.cuda.synchronize()

    x = qkv.clone().requires_grad_(True)
    ctx_ref, lse_ref = _ref(x, T, dh, keep)
    ctx_ref.backward(dctx)
    _, ctxd_ref = torch.autograd.functional.jvp(lambda y: _ref(y, T, dh, keep)[0], (qkv,), (qkvd,))

    tol = 2e-5 if dtype == torch.float32 else 3e-2

    def chk(name, got, want):
        err = (got.double().cpu() - want).abs().max().item()
        assert err <= tol * max(1.0, want.abs().max().item()), (name, err, want.abs().max().item())

    chk("ctx", ctx[:, :H], ctx_ref.detach())
    chk("lse", lse, lse_ref.detach())
    for t, name in enumerate(("dq", "dk", "dv")):
        chk(name, dqkv[:, t * H:(t + 1) * H], x.grad[:, t * H:(t + 1) * H])
    chk("ctx tangent", ctxd[:, :H], ctxd_ref)
    for name, t, cols in (("ctx", ctx, H), ("dqkv", dqkv, 3 * H), ("ctx tangent", ctxd, H)):
        assert torch.all(t[:, cols:] == SENT), f"{name}: written outside the head columns"
