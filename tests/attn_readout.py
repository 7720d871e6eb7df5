"""Test helper: read the attention-dropout mask straight out of a relative-attention forward kernel and compare it with
the host port of the mask hash (dropmask.py)."""
import torch

import dropmask as D
import txl_oracle as O

HS = 64


def shifted(x, off):
    """x's elements in a flat buffer starting `off` elements past an allocation (16- but not 32-byte aligned rows)."""
    buf = torch.zeros(off + x.numel(), device=x.device, dtype=x.dtype)
    buf[off:] = x.reshape(-1)
    return buf


def attn_readout(Q, M, dtype, impl, unaligned, p, seed, site, step=None):
    """Attention with q = k = r = u = vb = 0 and one-hot V rows (V[j] = e_j): output row i of head (b, n) is then
    keep_ij / ((1 - p) n_visible_i) on the visible keys, so its nonzero pattern is the kernel's dropout mask.  Checked
    against the host mask with the step counter value `step` (None: no counter); a wrong port and wrong arithmetic
    fail differently here.  unaligned: K / V base 16- but not 32-byte aligned (the generic kernels)."""
    from tgan_b200 import lib as L
    B, N, K, NH = 3, 5, M + Q, 5 * HS
    assert K <= HS
    z = lambda rows: torch.zeros(rows, NH, device="cuda", dtype=dtype)
    q, r = z(Q * B), z(K)
    kv = z(K * B).repeat(1, 2)
    vv = kv[:, NH:].view(K, B, N, HS)
    vv[torch.arange(K), :, :, torch.arange(K)] = 1
    off = 16 // kv.element_size() if unaligned else 0
    kvin = shifted(kv, off) if unaligned else kv
    u, vb = torch.zeros(NH, device="cuda"), torch.zeros(NH, device="cuda")
    reset = torch.tensor([0, 1, 0], dtype=torch.uint8, device="cuda")
    out = torch.empty(Q * B, NH, device="cuda", dtype=dtype)
    lse = torch.empty(B * N * Q, device="cuda")
    L.relattn_fwd(q, kvin, kvin, 2 * NH, r, u, vb, reset, out, lse, B, N, Q, M, Q, False, 0.125, p, seed, site,
                  impl=impl, k_off=off, v_off=off + NH)
    torch.cuda.synchronize()
    got = out.float().cpu().view(Q, B, N, HS).permute(1, 2, 0, 3)[..., :K].double()  # [B, N, Q, K]
    vis = ~O.attn_mask(Q, M, M, False, reset.cpu(), B)[:, None]                    # [B, 1, Q, K]
    keep = torch.from_numpy(D.attn_keep(seed, site, B, N, Q, K, p, step)) & vis
    want = keep.double() / ((1 - p) * vis.sum(-1, keepdim=True))
    assert torch.equal(got != 0, keep), f"mask differs at {(got != 0).ne(keep).sum().item()} of {keep.numel()} entries"
    assert (got - want).abs().max().item() <= 1e-2 * want.max().item()
    assert torch.all(out.float().view(Q * B, N, HS)[..., K:] == 0)
