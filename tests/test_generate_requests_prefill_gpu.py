"""GPU: generation from a request queue with one context pass per group of prompts
(MemTransformerLM.generate_requests(context_pass=True), tgan_ring_scatter, tgan_sample_step's run0).  Each request's
prefilled rows are copied into its column right below the write position of its first step, so every request
generates what generate_batched generates for it alone, whatever its prompt length and same_length."""
import weakref

import pytest
import torch

import mem_transformer as MT
import txl_oracle as O
from tgan_b200 import lib as L
from test_generate_requests_gpu import EMPTY, SETTINGS, V, _tiny
from test_model_gpu import build

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ring_scatter_is_bit_exact_and_touches_nothing_else(dtype):
    """Slabs [S][pos][col][DP] and K/V layers of the temporary layout [layer][pos * G + col][KW] from a 3-column source
    into a 5-column destination: a descriptor that fills the whole window, one with 0 rows, destination columns 0 and
    B - 1; the table is read from an offset.  Every other destination element keeps its sentinel."""
    g = torch.Generator().manual_seed(2)
    S, NL, DP, KW = 3, 2, 128, 192
    G, Cs, B, Cd, dst_end = 3, 11, 5, 17, 9
    src_x = torch.randn(S, Cs, G, DP, generator=g).to(dtype)
    src_kv = torch.randn(NL, Cs * G, KW, generator=g).to(dtype)
    dst_x = torch.full((S, Cd, B, DP), 7.0, dtype=dtype)
    dst_kv = torch.full((NL, Cd, B, KW), -3.0, dtype=dtype)
    desc = [[9, 9, 9, 9],  # not applied: the launch starts at descriptor 1
            [0, 2, 0, dst_end], [1, 4, 2, 0], [2, 5, B - 1, 3], [1, 7, 3, 4]]
    dx, dkv = dst_x.cuda(), dst_kv.cuda()
    L.ring_scatter(torch.tensor(desc, dtype=torch.int32).cuda(), 4, dst_end, dst_end, src_x.cuda(), dx, src_kv.cuda(),
                   dkv, src_kv_stride=Cs * G * KW, dst_kv_stride=Cd * B * KW, desc_off=1)
    want_x, want_kv = dst_x.clone(), dst_kv.clone()
    skv = src_kv.view(NL, Cs, G, KW)
    for sc, sp, dc, n in desc[1:]:
        want_x[:, dst_end - n:dst_end, dc] = src_x[:, sp:sp + n, sc]
        want_kv[:, dst_end - n:dst_end, dc] = skv[:, sp:sp + n, sc]
    assert torch.equal(dx.cpu(), want_x)
    assert torch.equal(dkv.cpu(), want_kv)
    assert (want_x[:, :, 1] == 7.0).all() and (want_x[:, dst_end:] == 7.0).all()  # the sentinel survives somewhere


LENS = [3, 9, 1, 30, 13, 7, 25, 2, 19]      # group 0 (longest prompt 9: K/V from the prefill ring's cache), groups
GENS = [40, 33, 25, 12, 28, 60, 17, 45, 50]  # 1 and 2 longer; prompts 30, 25, 19 exceed mem_len + 2 = 14


def _requests(g):
    prompts = [torch.randint(2, V, (n,), generator=g) for n in LENS]
    prompts[3][-2:] = EMPTY  # k = 2 (SETTINGS[3]): run0 = 1, the first sample is suppressed
    prompts[5][-3:] = EMPTY  # k = 1 (SETTINGS[5])
    prompts[7][-1] = EMPTY   # k = 1 (SETTINGS[7]): a two-token prompt whose last token is empty
    return [MT.GenRequest(p, n, empty_token=EMPTY, **s) for p, n, s in zip(prompts, GENS, SETTINGS)]


@pytest.mark.parametrize("same_length", [True, False])
def test_context_pass_requests_match_generate_py_for_every_prompt_length(same_length):
    """fp32 against generate.py restated with the oracle (its context pass over prompt[:-1], then single-token steps),
    per request alone, under the same injected uniforms (margin rule of test_ragged_generate_gpu): 9 requests on 3
    columns, every prompt length through the context pass, several ring re-layouts, requests that start on a window
    full of their predecessor's rows, and empty-bar suppression triggered by prompt-final empty tokens."""
    shape, model, params = _tiny(same_length)
    g = torch.Generator().manual_seed(9)
    reqs = _requests(g)
    U = [torch.rand(q.gen_len, generator=g) for q in reqs]
    out = model.generate_requests(reqs, 3, uniforms=U, context_pass=True)
    torch.cuda.synchronize()
    ml = shape.mem_len
    sch = MT.request_schedule([q.prompt.tolist() for q in reqs], GENS, 3, context_pass=True, mem_len=ml)
    S, B = sch.tables.shape[1:]
    assert S > 3 * (2 * ml + 1)  # the decode ring holds 2 * mem_len + 1 rows: several re-layouts
    assert max(LENS[:3]) - 1 <= 8 < min(max(LENS[3:6]), max(LENS[6:])) - 1  # both K/V paths of the prefill
    # some request starts while the window is full of the previous request of its column
    assert any(int(sch.start[t, c]) == t and int(sch.req[t - 1, c]) >= 0 and t - int(sch.start[t - 1, c]) >= ml
               for t in range(1, S) for c in range(B))
    checked = total = suppressed = 0
    for r, q in enumerate(reqs):
        got_r = out[r].cpu()
        assert got_r.dtype == torch.int64 and got_r.shape == (q.gen_len,)
        seq = q.prompt.tolist()
        om = None
        if len(seq) > 1:
            _, om = O.generate_logits(q.prompt[:-1].view(-1, 1), None, params, shape)
        k = q.num_empty_tokens_to_ignore
        for t in range(q.gen_len):
            lg, om = O.generate_logits(torch.tensor([[seq[-1]]]), om, params, shape)
            sup = k > 0 and len(seq) >= k and all(s == EMPTY for s in seq[-k:])
            suppressed += int(sup and t == 0)
            probs = O.generation_probs(lg[-1, 0], temperature=q.temperature, technique=q.technique, topk=q.topk,
                                       p=q.top_p, exclude_bos=q.exclude_bos, suppress_empty=sup, empty_bar_token=EMPTY)
            tok, margin = O.categorical_from_uniform(probs, float(U[r][t]))
            got = int(got_r[t])
            if margin < 2e-4:  # u within the fp32 model error of a CDF step: either neighbour is a legitimate draw
                assert probs[got] > 0, (r, t, got)
            else:
                assert got == tok, (r, t, got, tok, margin)
                checked += 1
            total += 1
            seq.append(got)
    assert checked > 0.85 * total, (checked, total)
    assert suppressed >= 3  # the prompt-final runs suppress the first sample of requests 3, 5 and 7


def test_one_prefill_ring_at_a_time_released_after_its_group_s_last_copy():
    """A group's prefill ring lives from its pass to the step of its group's last row copies: at most one is alive at
    any step, and none after the last copies of the queue.  The rings are sized for their own rows."""
    shape, model, _ = _tiny(True)
    eng = model._get_engine()
    reqs = _requests(torch.Generator().manual_seed(9))
    sch = MT.request_schedule([q.prompt.tolist() for q in reqs], GENS, 3, context_pass=True, mem_len=shape.mem_len)
    pl = sch.prefill
    last = {}
    for t, sl in pl.slices.items():
        for g, *_ in sl:
            last[g] = max(last.get(g, t), t)
    rings, orig = [], MT.MemTransformerLM._prefill_pass

    def spy(eng_, blk, pad):
        ctx = orig(model, eng_, blk, pad)
        rings.append(weakref.ref(ctx.ring.slabs))
        # sized for its own rows: a pass without memory needs no more than min(mem_len, Tm) of them
        Tm, ml = blk.shape[0], min(shape.mem_len, blk.shape[0])
        assert ctx.ring.capacity == (ml + Tm if Tm > eng.kv_cache_max_q else 2 * ml + Tm)
        return ctx

    model._prefill_pass = spy
    fd = sch.forced.clone()
    fd[fd < 0] = 5
    fd = fd.long().cuda()
    S = fd.shape[0]
    with torch.no_grad():
        cur = fd[0:1].clone()
        for t, _ in model._queue_forwards(eng, sch, sch.key_start.cuda(), cur, lambda x: x.cuda()):
            alive = [i for i, r in enumerate(rings) if r() is not None]
            assert len(alive) <= 1, (t, alive)
            assert all(t < last[i] for i in alive), (t, alive)  # released at the step of its group's last copies
            if t + 1 < S:
                cur.copy_(fd[t + 1:t + 2])
    assert len(rings) == sum(s is not None for s in pl.steps) == 3


def test_bf16_real_size_context_pass_matches_single_runs():
    """bf16 at the real model size (6 x 500, mem_len 128), prompts up to 240 tokens: 12 requests on 4 columns through
    the queue's prefill passes, copies and forwards, teacher-forced tokens in place of the samples.  Groups 0 and 2
    prefill on the tcgen05 forward with a key floor, group 1 (prompts <= 9 tokens) on the K/V-cache path.  Each
    request's logits at its first outputs match a B = 1 generate_batched + forward_generate run of it alone."""
    shape = O.TxlShape(n_layer=6, n_head=10, d_model=500, d_inner=1000, n_token=V, mem_len=128, same_length=True)
    model = build(shape, 5, 1, torch.bfloat16).eval()
    eng = model._get_engine()
    g = torch.Generator().manual_seed(4)
    lens = [200, 1, 33, 150, 5, 9, 2, 7, 181, 240, 17, 129]
    gens = [4, 9, 3, 6, 40, 3, 11, 5, 3, 7, 60, 4]
    prompts = [torch.randint(2, V, (n,), generator=g) for n in lens]
    C = 3  # outputs checked per request
    sch = MT.request_schedule([p.tolist() for p in prompts], gens, 4, context_pass=True, mem_len=shape.mem_len)
    forced = sch.forced.clone()
    teach = forced == -1
    forced[teach] = torch.randint(2, V, (int(teach.sum()),), generator=g, dtype=torch.int32)
    S, B = forced.shape
    fd = forced.long().cuda()
    got = {}
    with torch.no_grad():
        cur = fd[0:1].clone()
        for t, ectx in model._queue_forwards(eng, sch, sch.key_start.cuda(), cur, lambda x: x.cuda()):
            for c in range(B):
                r, off = int(sch.req[t, c]), int(sch.out_off[t, c])
                if r >= 0 and 0 <= off - sch.out_base[r] < C:
                    got[(r, off - sch.out_base[r])] = ectx.logits[c, :V].clone()
            if t + 1 < S:
                cur.copy_(fd[t + 1:t + 2])
        for r, p in enumerate(prompts):
            t0, c = (sch.req == r).nonzero()[0].tolist()
            _, m1 = model.generate_batched(p.view(-1, 1).cuda(), 0)
            steps = [int(p[-1])] + [int(forced[t0 + j, c]) for j in range(1, gens[r])]
            for j in range(min(C, gens[r])):
                lg, m1 = model.forward_generate(torch.tensor([[steps[j]]]).cuda(), m1)
                want, have = lg[0, 0, :V].float(), got[(r, j)]
                # 1e-2 of the values' scale (test_bf16_real_size_requests_match_single_runs): B = 4 and B = 1 round
                # differently in bf16; a missing, shifted or foreign prompt row moves them O(1)
                err = (have - want).abs().max().item()
                assert err <= 1e-2 * max(1.0, want.abs().max().item()), (r, j, err, want.abs().max().item())


def test_sample_step_run0_sets_the_run_at_a_start():
    """Argmax draws with the empty token on top, k = 3: a column whose request starts at this step begins its run at
    run0[request] instead of 0 and extends it by its input; other columns ignore run0.  run0 = NULL is run0 = 0."""
    E, k, step = EMPTY, 3, 8
    logits = torch.zeros(4, V)
    logits[:, E], logits[:, 11] = 50.0, 40.0
    settings = [(1, 32, 1, E, k, 0.0, 0.0)] * 3
    cur0 = [E, E, 5, E]
    start = [step, step, step, 2]   # columns 0-2 start requests 0-2, column 3 continues request 0
    run0 = torch.tensor([2, 1, 6], dtype=torch.int32, device="cuda")

    def step_with(r0):
        run = torch.tensor([0, 0, 0, 1], dtype=torch.int32, device="cuda")
        cur = torch.tensor(cur0, dtype=torch.int64, device="cuda")
        out = torch.full((4,), -9, dtype=torch.int64, device="cuda")
        probs = torch.full((4, V), -1.0, device="cuda")
        req_i = torch.tensor([s[:5] for s in settings], dtype=torch.int32).cuda()
        req_f = torch.tensor([s[5:] for s in settings], dtype=torch.float32).cuda()
        i32 = (lambda x: torch.tensor(x, dtype=torch.int32).cuda())
        L.sample_step(logits.cuda(), i32([0, 1, 2, 0]), i32(start), i32([0, 1, 2, 3]), None, req_i, req_f, run, cur,
                      out, V, step, run0=r0, probs_out=probs, seed=11, site=3)
        torch.cuda.synchronize()
        return run.cpu().tolist(), out.cpu().tolist(), probs.cpu()

    run, out, _ = step_with(run0)
    # col 0: 2 + E -> 3 >= k: suppressed; col 1: 1 + E -> 2; col 2: input 5 resets to 0; col 3: continues 1 + E -> 2
    assert run == [3, 2, 0, 2]
    assert out == [11, E, E, E]
    run_n, out_n, probs_n = step_with(None)
    run_z, out_z, probs_z = step_with(torch.zeros(3, dtype=torch.int32, device="cuda"))
    assert run_n == run_z == [1, 1, 0, 2] and out_n == out_z == [E, E, E, E]
    assert torch.equal(probs_n, probs_z)


def test_context_pass_with_device_rng_runs_without_host_sync():
    shape, model, _ = _tiny(True)
    g = torch.Generator().manual_seed(5)
    reqs = _requests(g)
    model.generate_requests(reqs[:2], 2, context_pass=True)  # engine creation and the parameter pack happen here
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = model.generate_requests(reqs, 3, context_pass=True)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    for q, o in zip(reqs, out):
        o = o.cpu()
        assert o.shape == (q.gen_len,) and ((o >= 0) & (o < V)).all()
        if q.exclude_bos:
            assert (o != 0).all()
        seq, k = q.prompt.tolist(), q.num_empty_tokens_to_ignore
        for tok in o.tolist():
            if k > 0 and len(seq) >= k and all(s == EMPTY for s in seq[-k:]):
                assert tok != EMPTY
            seq.append(tok)


def test_non_bool_context_pass_raises_before_any_launch():
    shape, model, _ = _tiny(True)
    p = torch.randint(2, V, (4,))
    ok = [MT.GenRequest(p, 3), MT.GenRequest(p[:1], 2)]
    n0 = L.launch_count()
    for bad in (1, 0, "yes", None, torch.tensor(True)):
        with pytest.raises(ValueError):
            model.generate_requests(ok, 2, context_pass=bad)
    assert L.launch_count() == n0
