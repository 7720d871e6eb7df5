"""GPU: every C-ABI kernel against a plain fp32 torch / oracle reference on seeded inputs."""
import math

import pytest
import torch

import dropmask as DM
from attn_readout import attn_readout

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _no_step_counter():
    """The host dropout masks assume no step counter; an earlier test may have registered the process-wide one."""
    with DM.pinned_step_counter(None):
        yield


def _keep(seed, site, rows, cols, ld, p, step=None):
    return torch.from_numpy(DM.elem_keep(seed, site, rows, cols, ld, p, step)).cuda()


def _lib():
    from tgan_b200 import lib
    return lib


def _rand(*shape, dtype=torch.float32, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to("cuda").to(dtype)


# ------------------------------------------------------------------------------------------------- GEMM
def _gemm_ref(A, B, transA, transB):
    a = A.float().t() if transA else A.float()
    b = B.float().t() if transB else B.float()
    return a @ b


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("transA,transB", [(False, True), (False, False), (True, False), (True, True)])
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 512, 512), (200, 310, 500 + 12), (129, 72, 40),
                                   (1000, 640, 1024), (64, 1280, 136)])
def test_gemm_layouts(impl, transA, transB, M, N, K):
    L = _lib()
    pad = lambda x: (x + 7) // 8 * 8
    A = _rand(*((K, pad(M)) if transA else (M, pad(K))), dtype=torch.bfloat16, seed=1)
    B = _rand(*((N, pad(K)) if transB else (K, pad(N))), dtype=torch.bfloat16, seed=2)
    Av = A[:, :M] if transA else A[:, :K]
    Bv = B[:, :K] if transB else B[:, :N]
    C = torch.full((M, pad(N) + 8), 7.0, device="cuda", dtype=torch.float32)
    L.gemm(A, B, C, transA=transA, transB=transB, M=M, N=N, K=K, impl=impl)
    torch.cuda.synchronize()
    ref = _gemm_ref(Av, Bv, transA, transB)
    err = (C[:, :N] - ref).abs().max().item()
    assert err <= 2e-3 * math.sqrt(K) , err
    assert torch.all(C[:, N:] == 7.0), "GEMM wrote outside its N columns"


@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("cdtype", [torch.float32, torch.bfloat16])
def test_gemm_epilogues(impl, cdtype):
    L = _lib()
    M, N, K = 300, 520, 320
    A, B = _rand(M, K, dtype=torch.bfloat16, seed=3), _rand(N, K, dtype=torch.bfloat16, seed=4)
    bias = _rand(N, seed=5)
    aux = _rand(M, N, dtype=torch.bfloat16, seed=6)
    aux32 = _rand(M, N, seed=7)
    ref0 = A.float() @ B.float().t()
    tol = 0.08 if cdtype == torch.bfloat16 else 0.02

    def run(flags, alpha=1.0, aux_t=None, C0=None, **kw):
        C = torch.zeros(M, N, device="cuda", dtype=cdtype) if C0 is None else C0.clone()
        L.gemm(A, B, C, M=M, N=N, K=K, bias=bias, aux=aux_t, ldaux=N, flags=flags, alpha=alpha, impl=impl, **kw)
        torch.cuda.synchronize()
        return C.float()

    assert (run(L.EPI_BIAS | L.EPI_RELU) - torch.relu(ref0 + bias)).abs().max() < tol * 4
    assert (run(L.EPI_ADD_AUX, alpha=0.5, aux_t=aux) - (0.5 * ref0 + aux.float())).abs().max() < tol * 4
    assert (run(L.EPI_ADD_AUX, aux_t=aux32) - (ref0 + aux32)).abs().max() < tol * 4
    got = run(L.EPI_MASK_POS, alpha=2.0, aux_t=aux)
    assert (got - torch.where(aux.float() > 0, 2.0 * ref0, torch.zeros_like(ref0))).abs().max() < tol * 8
    C0 = _rand(M, N, dtype=cdtype, seed=8)
    assert (run(L.EPI_ACCUM, C0=C0) - (ref0 + C0.float())).abs().max() < tol * 4
    # dropout: the host mask at element row * ldc + col, survivors scaled by 1/(1-p); also with a row pitch wider than N
    for ldc in (N, N + 24):
        C = torch.full((M, ldc), 7.0, device="cuda", dtype=cdtype)
        L.gemm(A, B, C, M=M, N=N, K=K, ldc=ldc, flags=L.EPI_DROPOUT, drop_p=0.25, seed=2 ** 35 + 11, site=5, impl=impl)
        torch.cuda.synchronize()
        keep, d = _keep(2 ** 35 + 11, 5, M, N, ldc, 0.25), C[:, :N].float()
        assert torch.all(d[~keep] == 0), "an element the mask drops survived"
        assert torch.all(d[keep & (ref0.abs() > 1)] != 0), "an element the mask keeps was dropped"
        assert ((d - ref0 / 0.75).abs() * keep).max() < tol * 6
        assert torch.all(C[:, N:] == 7.0)


def test_gemm_tc_large_k_accumulation_and_persistence():
    """wgrad-like shape: long K, more tiles than SMs, fp32 output."""
    L = _lib()
    M, N, K = 1280, 512, 8192
    A, B = _rand(K, M, dtype=torch.bfloat16, seed=9, scale=0.1), _rand(K, N, dtype=torch.bfloat16, seed=10, scale=0.1)
    C = torch.empty(M, N, device="cuda", dtype=torch.float32)
    L.gemm(A, B, C, transA=True, transB=False, M=M, N=N, K=K, impl=2)
    ref = A.float().t() @ B.float()
    assert (C - ref).abs().max().item() < 2e-2
    # split-K with accumulation onto an existing fp32 gradient, ragged N, row pitch wider than N
    C0 = _rand(M, N + 8, seed=21)
    C = C0.clone()
    L.gemm(A, B, C, transA=True, transB=False, M=M, N=N - 3, K=K, flags=L.EPI_ACCUM, alpha=0.5, impl=2)
    assert (C[:, :N - 3] - (C0[:, :N - 3] + 0.5 * ref[:, :N - 3])).abs().max().item() < 2e-2
    assert torch.equal(C[:, N - 3:], C0[:, N - 3:])
    M, N, K = 148 * 128 * 2 + 77, 256, 192
    A, B = _rand(M, K, dtype=torch.bfloat16, seed=11), _rand(N, K, dtype=torch.bfloat16, seed=12)
    C = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    L.gemm(A, B, C, M=M, N=N, K=K, impl=2)
    ref = A.float() @ B.float().t()
    assert (C.float() - ref).abs().max().item() < 0.3


@pytest.mark.parametrize("cdtype", [torch.bfloat16, torch.float32])
def test_gemm_tc_cta_pair_kernel(cdtype):
    """Shapes with >= 74 output tiles of 256 x 256 take the 2-CTA (cta_group::2) kernel: plain, fused FFN and residual
    epilogues, ragged M / N edges, and the dropout mask the host regenerates."""
    L = _lib()
    M, N, K = 4100, 1288, 520
    A, B = _rand(M, K, dtype=torch.bfloat16, seed=3, scale=0.5), _rand(N, K, dtype=torch.bfloat16, seed=4, scale=0.5)
    bias, aux = _rand(N, seed=5), _rand(M, N, dtype=torch.bfloat16, seed=6)
    ref0 = A.float() @ B.float().t()
    tol = 0.15 if cdtype == torch.bfloat16 else 0.02

    def run(flags, impl=2, **kw):
        C = torch.full((M, N), 7.0, device="cuda", dtype=cdtype)
        L.gemm(A, B, C, M=M, N=N, K=K, bias=bias, aux=aux, ldaux=N, flags=flags, impl=impl, **kw)
        torch.cuda.synchronize()
        return C.float()

    assert (run(0) - ref0).abs().max() < tol
    assert (run(L.EPI_BIAS | L.EPI_RELU) - torch.relu(ref0 + bias)).abs().max() < tol
    assert (run(L.EPI_ADD_AUX) - (ref0 + aux.float())).abs().max() < tol
    d = run(L.EPI_BIAS | L.EPI_RELU | L.EPI_DROPOUT, drop_p=0.25, seed=11, site=5)
    keep, want = _keep(11, 5, M, N, N, 0.25), torch.relu(ref0 + bias) / 0.75
    assert torch.all(d[~keep] == 0), "an element the mask drops survived"
    assert torch.all(d[keep & (want > 0.5)] != 0), "an element the mask keeps was dropped"
    assert ((d - want).abs() * keep).max() < tol / 0.75


def test_gemm_fp32_simt_exact():
    L = _lib()
    M, N, K = 77, 130, 500
    A, B = _rand(M, K, seed=13), _rand(N, K, seed=14)
    C = torch.empty(M, N, device="cuda")
    L.gemm(A, B, C, M=M, N=N, K=K)
    ref = (A.double() @ B.double().t()).float()
    assert (C - ref).abs().max().item() < 2e-4


# ------------------------------------------------------------------------------------------------- row ops
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_layernorm_fwd_bwd(dtype):
    L = _lib()
    rows, D, DP = 333, 500, 512
    z = _rand(rows, DP, seed=1)
    z[:, D:] = 0
    gamma, beta = torch.zeros(DP, device="cuda"), torch.zeros(DP, device="cuda")
    gamma[:D], beta[:D] = _rand(D, seed=2) * 0.1 + 1, _rand(D, seed=3) * 0.1
    y = torch.empty(rows, DP, device="cuda", dtype=dtype)
    mean, rstd = torch.empty(rows, device="cuda"), torch.empty(rows, device="cuda")
    L.ln_fwd(z, y, gamma, beta, mean, rstd, rows, D, DP)
    zr = z[:, :D].double().requires_grad_(True)
    ref = torch.nn.functional.layer_norm(zr, (D,), gamma[:D].double(), beta[:D].double())
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    assert (y[:, :D].double() - ref).abs().max() < tol
    assert torch.all(y[:, D:] == 0)
    y1 = torch.empty_like(y)
    L.ln_fwd(z, y1, gamma, beta, mean, rstd, rows, D, DP, pad_one=True)  # ones column in the first pad lane
    assert torch.equal(y1[:, :D], y[:, :D]) and torch.all(y1[:, D] == 1) and torch.all(y1[:, D + 1:] == 0)
    dy = _rand(rows, DP, dtype=dtype, seed=4)
    dz, dzd = torch.empty_like(dy), torch.empty_like(dy)
    dg, db = torch.zeros(DP, device="cuda"), torch.zeros(DP, device="cuda")
    dsum = torch.zeros(DP, device="cuda")
    L.ln_bwd(dy, z, gamma, mean, rstd, dz, dzd, dg, db, rows, D, DP, 0.2, 3, 9, dsum=dsum)
    # fused bias gradient: column sums of the dropped gradient (fp32 sums of the values before the bf16 store)
    assert (dsum[:D] - dzd[:, :D].float().sum(0)).abs().max() < (1e-4 if dtype == torch.float32 else 0.15)
    gref = gamma[:D].double().clone().requires_grad_(True)
    bref = beta[:D].double().clone().requires_grad_(True)
    out = torch.nn.functional.layer_norm(zr, (D,), gref, bref)
    out.backward(dy[:, :D].double())
    assert (dz[:, :D].double() - zr.grad).abs().max() < (1e-4 if dtype == torch.float32 else 3e-2)
    assert (dg[:D].double() - gref.grad).abs().max() < (1e-3 if dtype == torch.float32 else 0.2)
    assert (db[:D].double() - bref.grad).abs().max() < (1e-3 if dtype == torch.float32 else 0.2)
    # dz_drop: the host mask at element row * DP + col
    keep = _keep(3, 9, rows, D, DP, 0.2)
    assert torch.all(dzd[:, :D][~keep] == 0)
    assert torch.all(dzd[:, :D][keep & (dz[:, :D].abs() > 1e-3)] != 0)
    assert ((dzd[:, :D].float() - dz[:, :D].float() / 0.8).abs() * keep).max() < 3e-2


def test_embedding_and_posemb():
    L = _lib()
    V, D, DP, rows = 310, 500, 512, 257
    E = torch.zeros(320, DP, device="cuda")
    E[:V, :D] = _rand(V, D, seed=1)
    ids = torch.randint(0, V, (rows,), device="cuda")
    out = torch.empty(rows, DP, device="cuda")
    L.embed_fwd(ids, E, out, rows, D, DP, math.sqrt(D), 0.0, 0, 0)
    assert torch.allclose(out[:, :D], E[ids, :D] * math.sqrt(D), rtol=1e-6, atol=1e-6)
    assert torch.all(out[:, D:] == 0)
    dout = _rand(rows, DP, seed=2)
    dE = torch.zeros(320, DP, device="cuda")
    L.embed_bwd(ids, dout, dE, rows, V, D, DP, math.sqrt(D), 0.0, 0, 0)
    ref = torch.zeros(V, D, device="cuda", dtype=torch.float64)
    ref.index_add_(0, ids, dout[:, :D].double() * math.sqrt(D))
    assert (dE[:V, :D].double() - ref).abs().max() < 1e-3
    import txl_oracle as O
    K = 1152
    pe = torch.empty(K, DP, device="cuda")
    inv = (1 / (10000 ** (torch.arange(0.0, D, 2.0) / D))).cuda()
    L.pos_emb(inv, pe, K, D, DP, -1, 0.0, 0, 0)
    ref = O.positional_embedding(K, D)
    assert (pe[:, :D].cpu() - ref).abs().max() < 2e-4  # fp32 sin/cos of arguments up to 1151 rad
    L.pos_emb(inv, pe, K, D, DP, 100, 0.0, 0, 0)
    assert (pe[:, :D].cpu() - O.positional_embedding(K, D, 100)).abs().max() < 2e-4


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_elementwise_dropout_sites_match_host_mask(dtype):
    """tgan_dropout, embed_fwd, embed_bwd and pos_emb with dropout on: exactly the host mask at row * ld + col."""
    L = _lib()
    p, seed, site = 0.1, 2 ** 33 + 5, 2 ** 32 + 7
    rows, cols, lds, ldd = 301, 200, 216, 232
    src = _rand(rows, lds, dtype=dtype, seed=3)
    dst = torch.full((rows, ldd), 9.0, device="cuda", dtype=dtype)
    L.dropout(src, dst, rows, cols, lds, ldd, p, seed, site)
    keep = _keep(seed, site, rows, cols, ldd, p)
    want = torch.where(keep, src[:, :cols].float() / (1 - p), torch.zeros(()).cuda())
    tol = 1e-6 if dtype == torch.float32 else 1e-2
    assert ((dst[:, :cols].float() - want).abs() <= tol * want.abs()).all()
    assert torch.all(dst[:, cols:] == 9.0)

    V, D, DP, n = 310, 500, 512, 257
    E = torch.zeros(320, DP, device="cuda", dtype=dtype)
    E[:V, :D] = _rand(V, D, seed=1, dtype=dtype)
    ids = torch.randint(0, V, (n,), device="cuda")
    out = torch.empty(n, DP, device="cuda", dtype=dtype)
    L.embed_fwd(ids, E, out, n, D, DP, math.sqrt(D), p, seed, site)
    keep = _keep(seed, site, n, D, DP, p)
    want = torch.where(keep, E[ids, :D].float() * (math.sqrt(D) / (1 - p)), torch.zeros(()).cuda())
    assert ((out[:, :D].float() - want).abs() <= 1e-5 + tol * want.abs()).all()
    assert torch.all(out[:, D:] == 0)

    dout = _rand(n, DP, dtype=dtype, seed=2)
    dE = torch.zeros(320, DP, device="cuda")
    L.embed_bwd(ids, dout, dE, n, V, D, DP, math.sqrt(D), p, seed, site)
    ref = torch.zeros(V, D, device="cuda", dtype=torch.float64)
    ref.index_add_(0, ids, dout[:, :D].double() * keep * (math.sqrt(D) / (1 - p)))
    assert (dE[:V, :D].double() - ref).abs().max() < 1e-3

    K = 300
    pe = torch.empty(K, DP, device="cuda", dtype=dtype)
    pe0 = torch.empty(K, DP, device="cuda", dtype=dtype)
    inv = (1 / (10000 ** (torch.arange(0.0, D, 2.0) / D))).cuda()
    L.pos_emb(inv, pe0, K, D, DP, -1, 0.0, 0, 0)
    L.pos_emb(inv, pe, K, D, DP, -1, p, seed, site)
    keep = _keep(seed, site, K, D, DP, p)
    want = torch.where(keep, pe0[:, :D].float() / (1 - p), torch.zeros(()).cuda())
    assert ((pe[:, :D].float() - want).abs() <= 1e-6 + tol * want.abs()).all()
    assert torch.all(pe[:, D:] == 0)


def test_step_counter_folds_into_the_masks():
    """With a registered step counter every mask key becomes mix32(key ^ counter * 0x9E3779B1) (common.cuh step_fold):
    an element-wise mask and an attention mask follow the host port with the same counter value, and differ from the
    masks without it."""
    L = _lib()
    rows, cols, p = 64, 256, 0.25
    ones = torch.ones(rows, cols, device="cuda")
    with DM.pinned_step_counter(977):
        m = torch.empty_like(ones)
        L.dropout(ones, m, rows, cols, cols, cols, p, 5, 6)
        torch.cuda.synchronize()
        assert torch.equal(m != 0, _keep(5, 6, rows, cols, cols, p, step=977))
        assert not torch.equal(m != 0, _keep(5, 6, rows, cols, cols, p))
        attn_readout(16, 30, torch.float32, 1, False, p, 7, 8, step=977)
    # on exit the process-wide counter (if one was created) is registered again
    ctr = L._step_counters.get(torch.cuda.current_device())
    m0 = torch.empty_like(ones)
    L.dropout(ones, m0, rows, cols, cols, cols, p, 5, 6)
    torch.cuda.synchronize()
    step = None if ctr is None else int(ctr.item())
    assert torch.equal(m0 != 0, _keep(5, 6, rows, cols, cols, p, step=step))


def test_cross_entropy_and_gumbel():
    L = _lib()
    import txl_oracle as O
    rows, V, VP = 515, 310, 320
    logits = _rand(rows, VP, seed=1, scale=3.0)
    tgt = torch.randint(0, V, (rows,), device="cuda")
    nll, lse = torch.empty(rows, device="cuda"), torch.empty(rows, device="cuda")
    L.ce_fwd(logits, tgt, nll, lse, rows, V)
    lr = logits[:, :V].double().requires_grad_(True)
    ref = torch.nn.functional.cross_entropy(lr, tgt, reduction="none")
    assert (nll.double() - ref).abs().max() < 1e-5
    dn = _rand(rows, seed=2)
    dl = torch.empty(rows, VP, device="cuda")
    L.ce_bwd(logits, tgt, lse, dn, dl, rows, V, VP)
    ref.backward(dn.double())
    assert (dl[:, :V].double() - lr.grad).abs().max() < 1e-5
    assert torch.all(dl[:, V:] == 0)
    # gumbel straight-through with injected noise vs the oracle restatement (mem_transformer.py:609-628)
    for tau in (1.0, 0.05):
        U = torch.rand(rows, V, generator=torch.Generator().manual_seed(5)).cuda()
        y, st = torch.empty(rows, V, device="cuda"), torch.empty(rows, V, device="cuda")
        ids = torch.empty(rows, dtype=torch.int64, device="cuda")
        L.gumbel_st_fwd(logits, U, tau, y, st, ids, rows, V)
        st_ref, y_ref, ids_ref = O.gumbel_st(logits[:, :V].cpu(), U.cpu(), tau)
        # bit-exact ids wherever the top-2 margin of the perturbed logits is not a rounding tie
        z = (logits[:, :V].cpu().double() + O.gumbel_noise(U.cpu().double()))
        top2 = z.topk(2, dim=-1).values
        clear = (top2[:, 0] - top2[:, 1]) > 1e-4
        assert clear.float().mean() > 0.99
        assert torch.equal(ids.cpu()[clear], ids_ref[clear])
        assert (y.cpu() - y_ref).abs().max() < 2e-5
        assert (st.cpu()[clear] - st_ref[clear]).abs().max() < 1e-6
        dst = _rand(rows, V, seed=6)
        dlg = torch.empty(rows, V, device="cuda")
        L.gumbel_st_bwd(y, dst, tau, dlg, rows, V)
        ref = (1 / tau) * y * (dst - (y * dst).sum(-1, keepdim=True))
        assert (dlg - ref).abs().max() < 1e-4 / tau
    # device-side noise: uniform argmax frequencies follow softmax(logits) roughly
    big = torch.zeros(20000, VP, device="cuda")
    big[:, 3] = 1.0
    y = torch.empty(20000, V, device="cuda")
    ids = torch.empty(20000, dtype=torch.int64, device="cuda")
    L.gumbel_st_fwd(big, None, 1.0, y, None, ids, 20000, V, seed=123, site=1)
    p3 = math.e / (math.e + V - 1)
    assert abs((ids == 3).float().mean().item() - p3) < 0.004


def test_colsum_convert_dropout_pack_adam():
    L = _lib()
    x = _rand(1000, 520, dtype=torch.bfloat16, seed=1)
    out = torch.ones(520, device="cuda")
    L.colsum(x, out, 1000, 500)
    assert (out[:500] - 1 - x[:, :500].float().sum(0)).abs().max() < 1e-2
    assert torch.all(out[500:] == 1)
    src = _rand(37, 50, seed=2)
    dst = torch.full((37, 64), 9.0, device="cuda", dtype=torch.bfloat16)
    L.convert(src, 50, dst, 64, 37, 50, 64)
    assert torch.equal(dst[:, :50], src.bfloat16()) and torch.all(dst[:, 50:] == 0)
    # pack: [3*N*dh, D] qkv weight -> head-padded rows, plus the transposed copy; unpack inverts it
    N, dh, D, DP = 4, 10, 40, 64
    W = _rand(3 * N * dh, D, seed=3)
    u = _rand(N, dh, seed=4)
    mat = torch.zeros(2 * 3 * N * 64 * DP, device="cuda", dtype=torch.bfloat16)
    vec = torch.zeros(N * 64, device="cuda")
    rows = [[W.data_ptr(), 0, 3 * N * dh, D, DP, dh, 64, 1, 1, 0, 0, 0],
            [W.data_ptr(), 3 * N * 64 * DP, 3 * N * dh, D, 3 * N * 64, dh, 64, 1, 1, 1, 0, 0],
            [u.data_ptr(), 0, 1, N * dh, N * dh, 1, 1, dh, 64, 0, 1, 0]]
    desc = torch.tensor(rows, dtype=torch.int64, device="cuda")
    L.pack_params(mat, vec, desc, 3, W.numel())
    P = mat[:3 * N * 64 * DP].view(3 * N, 64, DP)
    assert torch.equal(P[:, :dh, :D], W.bfloat16().view(3 * N, dh, D))
    assert torch.all(P[:, dh:, :] == 0) and torch.all(P[:, :, D:] == 0)
    PT = mat[3 * N * 64 * DP:].view(DP, 3 * N * 64)
    assert torch.equal(PT.t().contiguous().view(3 * N, 64, DP), P)
    assert torch.equal(vec.view(N, 64)[:, :dh], u)
    g = torch.empty_like(W)
    gm = P.float().contiguous().view(-1)
    L.unpack_grads(gm, vec, torch.tensor([[g.data_ptr()] + rows[0][1:]], dtype=torch.int64, device="cuda"), 1, W.numel())
    assert torch.equal(g, W.bfloat16().float())
    # fused clip + Adam vs torch.optim.Adam after clip_grad_norm_
    p0, g0 = _rand(5000, seed=5), _rand(5000, seed=6)
    pr = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([pr], lr=1e-2)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    nsq = torch.zeros(1, device="cuda")
    for step in range(1, 4):
        pr.grad = g0.clone() * step
        torch.nn.utils.clip_grad_norm_([pr], 3.0)
        opt.step()
        nsq.zero_()
        L.sumsq(g0 * step, 5000, nsq)
        L.adam_step(p, g0 * step, m, v, 5000, 1e-2, 0.9, 0.999, 1e-8, 0.0, step, nsq, 3.0, 1.0)
    assert (p - pr.detach()).abs().max() < 1e-5


@pytest.mark.parametrize("M,K,N,bias", [(640, 310, 64, False), (512, 1200, 1200, True), (384, 1200, 100, True)])
def test_nn_linear_forward_backward_match_torch(M, K, N, bias):
    """tgan_b200.nn.linear (RelGAN_D's dense layers on tgan_gemm: forward, dgrad, wgrad, bias gradient) against
    F.linear in fp64 on bf16-rounded operands; shapes = the discriminator's three layers (vocabulary 310 -> padded)."""
    from tgan_b200.nn import linear
    g = torch.Generator().manual_seed(M + N)
    x = torch.randn(M, K, generator=g).bfloat16().float().cuda().requires_grad_(True)
    w = (0.05 * torch.randn(N, K, generator=g)).bfloat16().float().cuda().requires_grad_(True)
    b = (0.1 * torch.randn(N, generator=g)).cuda().requires_grad_(True) if bias else None
    y = linear(x, w, b)
    dy = torch.randn(M, N, generator=g).bfloat16().float().cuda()
    y.backward(dy)
    xd, wd = x.detach().double(), w.detach().double()
    yr = xd @ wd.t() + (b.detach().double() if bias else 0)
    assert (y.double() - yr).abs().max() < 2e-3 * yr.abs().max()
    dxr, dwr = dy.double() @ wd, dy.double().t() @ xd
    assert (x.grad.double() - dxr).abs().max() < 2e-3 * dxr.abs().max()
    assert (w.grad.double() - dwr).abs().max() < 2e-3 * dwr.abs().max()
    if bias:
        assert (b.grad.double() - dy.double().sum(0)).abs().max() < 1e-3 * dy.abs().sum(0).max()
