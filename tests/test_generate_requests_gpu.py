"""GPU: generation from a request queue (MemTransformerLM.generate_requests, tgan_sample_step).  A column that finishes
a request takes the next one inside the same ring memory; the per-sequence key floor hides the earlier requests'
rows, so every request generates what it generates alone."""
import pytest
import torch

import mem_transformer as MT
import txl_oracle as O
from tgan_b200 import lib as L
from test_model_gpu import build

pytestmark = pytest.mark.gpu
V = 310
EMPTY = 37  # the empty-bar token of every request here; its output bias is raised so that runs of it occur


def _tiny(same_length, seed=31):
    shape = O.TxlShape(n_layer=2, n_head=4, d_model=40, d_inner=72, n_token=V, mem_len=12, same_length=same_length)
    model = build(shape, seed, 1, torch.float32).eval()
    with torch.no_grad():
        model.crit.out_layers[0].bias[EMPTY] += 6.0
    params = {k: v.double() for k, v in O.init_params(shape, seed).items()}
    params["crit.out_layers.0.bias"] = params["crit.out_layers.0.bias"].clone()
    params["crit.out_layers.0.bias"][EMPTY] += 6.0
    return shape, model, params


SETTINGS = [
    dict(technique="topk", topk=32, temperature=0.95),
    dict(technique="nucleus", top_p=0.9, temperature=1.0),
    dict(technique="random", temperature=0.8, exclude_bos=False),
    dict(technique="topk", topk=6, temperature=0.95, num_empty_tokens_to_ignore=2),
    dict(technique="topk", topk=8, temperature=0.0),
    dict(technique="nucleus", top_p=0.5, temperature=0.9, exclude_bos=False, num_empty_tokens_to_ignore=1),
    dict(technique="random", temperature=1.1, num_empty_tokens_to_ignore=3),
    dict(technique="topk", topk=32, temperature=0.95, num_empty_tokens_to_ignore=1),
    dict(technique="topk", topk=1, temperature=0.7),
]
LENS = [30, 1, 13, 7, 2, 25, 14, 1, 19]
GENS = [12, 40, 1, 33, 25, 5, 17, 28, 9]


def _requests(g, lens=LENS, gens=GENS, settings=SETTINGS):
    prompts = [torch.randint(2, V, (n,), generator=g) for n in lens]
    prompts[3][-2:] = EMPTY  # a run of k = 2 at the end of the prompt: the first sample is suppressed
    prompts[7][-1] = EMPTY   # a one-token prompt that is a run of k = 1
    return [MT.GenRequest(p, n, empty_token=EMPTY, **s) for p, n, s in zip(prompts, gens, settings)]


@pytest.mark.parametrize("same_length", [True, False])
def test_requests_match_generate_py_for_each_request_alone(same_length):
    """fp32 against generate.py restated with the oracle, per request on its own prompt, under the same injected
    uniforms (margin rule of test_ragged_generate_gpu).  9 requests on 3 columns: the columns are refilled several
    times, the ring is re-laid out many times and a request starts on a window full of its predecessor's rows.
    With same_length=False a prompt row of the one-token prefill sees at most mem_len earlier rows, so the oracle feeds
    prompts longer than mem_len + 2 one token at a time (shorter ones: generate.py's context pass, which equals it)."""
    shape, model, params = _tiny(same_length)
    g = torch.Generator().manual_seed(9)
    reqs = _requests(g)
    U = [torch.rand(q.gen_len, generator=g) for q in reqs]
    out = model.generate_requests(reqs, 3, uniforms=U)
    torch.cuda.synchronize()
    sch = MT.request_schedule([q.prompt.tolist() for q in reqs], GENS, 3)
    S, B = sch.tables.shape[1:]
    assert S > 3 * (2 * shape.mem_len + 1)  # the decode ring holds 2 * mem_len + 1 rows: several re-layouts
    # some request starts while the window is full of the previous request of its column
    assert any(int(sch.key_start[t, c]) == t and t >= shape.mem_len and int(sch.key_start[t - 1, c]) <= t - shape.mem_len
               and int(sch.req[t - 1, c]) >= 0 for t in range(1, S) for c in range(B))
    checked = total = suppressed = 0
    for r, q in enumerate(reqs):
        got_r = out[r].cpu()
        assert got_r.dtype == torch.int64 and got_r.shape == (q.gen_len,)
        seq = q.prompt.tolist()
        om = None
        if same_length or len(seq) <= shape.mem_len + 2:
            if len(seq) > 1:
                _, om = O.generate_logits(q.prompt[:-1].view(-1, 1), None, params, shape)
        else:
            for tok in seq[:-1]:
                _, om = O.generate_logits(torch.tensor([[tok]]), om, params, shape)
        k = q.num_empty_tokens_to_ignore
        for t in range(q.gen_len):
            lg, om = O.generate_logits(torch.tensor([[seq[-1]]]), om, params, shape)
            sup = k > 0 and len(seq) >= k and all(s == EMPTY for s in seq[-k:])
            suppressed += int(sup)
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
    assert suppressed > 0


def test_bf16_real_size_requests_match_single_runs():
    """bf16 at the real model size (6 x 500, mem_len 128): 12 requests on 4 columns, run through the schedule's
    forwards with the key floor and teacher-forced tokens in place of the samples.  Each request's logits at its
    first outputs match a B = 1 run of that request alone (context pass over the prompt, then single-token steps)."""
    shape = O.TxlShape(n_layer=6, n_head=10, d_model=500, d_inner=1000, n_token=V, mem_len=128, same_length=True)
    model = build(shape, 5, 1, torch.bfloat16).eval()
    eng = model._get_engine()
    g = torch.Generator().manual_seed(4)
    lens = [200, 1, 33, 150, 5, 97, 64, 181, 2, 129, 17, 240]
    gens = [4, 9, 3, 6, 40, 3, 11, 5, 3, 7, 60, 4]
    prompts = [torch.randint(2, V, (n,), generator=g) for n in lens]
    C = 3  # outputs checked per request
    sch = MT.request_schedule([p.tolist() for p in prompts], gens, 4)
    forced = sch.forced.clone()
    teach = forced == -1
    forced[teach] = torch.randint(2, V, (int(teach.sum()),), generator=g, dtype=torch.int32)
    S, B = forced.shape
    assert S > 2 * (shape.mem_len + 1)  # the window re-lays out and slides across request boundaries
    fd, ks = forced.long().cuda(), sch.key_start.cuda()
    got = {}
    with torch.no_grad():
        mems = eng.new_ring(B, 1, shape.mem_len)
        for t in range(S):
            mems.key_start = ks[t]
            ectx = eng.forward(fd[t:t + 1], None, mems, mem_len=shape.mem_len, same_length=True, training=False,
                               save_for_backward=False)
            mems = ectx.new_mems
            for c in range(B):
                r, off = int(sch.req[t, c]), int(sch.out_off[t, c])
                if r >= 0 and 0 <= off - sch.out_base[r] < C:
                    got[(r, off - sch.out_base[r])] = ectx.logits[c, :V].clone()

        for r, p in enumerate(prompts):
            t, c = (sch.req == r).nonzero(as_tuple=True)
            t0, c = int(t[0]), int(c[0])
            T = len(p)
            _, m1 = model.generate_batched(p.view(-1, 1).cuda(), 0)
            steps = [int(p[-1])] + [int(forced[t0 + T + j, c]) for j in range(gens[r] - 1)]
            for j in range(min(C, gens[r])):
                lg, m1 = model.forward_generate(torch.tensor([[steps[j]]]).cuda(), m1)
                want, have = lg[0, 0, :V].float(), got[(r, j)]
                # 1e-2 of the values' scale (test_ragged_bf16_real_size_matches_single_prompt_runs): B = 4 and B = 1
                # round differently in bf16; a row of the previous request leaking into the attention moves them O(1)
                err = (have - want).abs().max().item()
                assert err <= 1e-2 * max(1.0, want.abs().max().item()), (r, j, err, want.abs().max().item())


def _sample_step(logits, req, start, out_off, forced_next, settings, run, cur, out, step, u=None, probs=None):
    req_i = torch.tensor([s[:5] for s in settings], dtype=torch.int32).cuda()
    req_f = torch.tensor([s[5:] for s in settings], dtype=torch.float32).cuda()
    i32 = (lambda x: None if x is None else torch.tensor(x, dtype=torch.int32).cuda())
    L.sample_step(logits, i32(req), i32(start), i32(out_off), i32(forced_next), req_i, req_f, run, cur, out, V, step,
                  u=u, probs_out=probs, seed=11, site=3)


def test_sample_step_matches_sample_tokens_per_setting():
    """Per column: the request's settings, its empty-bar run, the draw on u[out_off], the sample into out[out_off] and
    the next input; ids and filtered distributions equal tgan_sample_tokens called once per setting, bit for bit."""
    g = torch.Generator().manual_seed(1)
    # (mode, topk, exclude_bos, empty_token, k, temperature, top_p)
    settings = [(1, 32, 1, 101, 0, 0.95, 0.0), (1, 5, 0, 101, 1, 1.3, 0.0), (2, 0, 1, 101, 1, 0.9, 0.9),
                (0, 0, 1, 7, 2, 1.0, 0.0), (1, 32, 0, 101, 1, 0.0, 0.0), (2, 0, 0, 7, 0, 1.1, 0.4)]
    R, step = len(settings), 5
    busy, idle = 4 * R, 3
    B = busy + idle
    logits = (3.0 * torch.randn(B, 320, generator=g)).cuda()
    req = [b % R for b in range(busy)] + [-1] * idle
    cur0 = [settings[b % R][3] if (b // R) % 2 else 5 for b in range(busy)] + [9] * idle
    forced_next = [-1 if b % 2 == 0 else 100 + b for b in range(busy)] + [7] * idle
    out_off = list(range(busy)) + [-1] * idle
    u = torch.rand(B, generator=g).cuda()
    run = torch.full((B,), 4, dtype=torch.int32, device="cuda")  # every busy column starts a request: reset to 0
    cur = torch.tensor(cur0, dtype=torch.int64).cuda()
    out = torch.full((busy,), -9, dtype=torch.int64, device="cuda")
    probs = torch.full((B, V), -1.0, device="cuda")
    _sample_step(logits, req, [step] * B, out_off, forced_next, settings, run, cur, out, step, u=u, probs=probs)

    want_run = torch.tensor([int(cur0[b] == settings[b % R][3]) for b in range(busy)] + [4] * idle, dtype=torch.int32)
    want_ids = torch.empty(busy, dtype=torch.int64)
    want_probs = torch.empty(busy, V)
    for i, (mode, topk, xb, e, k, temp, top_p) in enumerate(settings):
        rows = torch.tensor([b for b in range(busy) if req[b] == i])
        sup = ((want_run[rows] >= k) & (k > 0)).to(torch.uint8).cuda()
        ids = torch.empty(len(rows), dtype=torch.int64, device="cuda")
        pr = torch.empty(len(rows), V, device="cuda")
        L.sample_tokens(logits[rows.cuda()], ids, V, u=u[rows.cuda()].contiguous(), suppress_empty=sup, probs_out=pr,
                        exclude_bos=bool(xb), empty_token=e, mode=mode, topk=topk, top_p=top_p, temperature=temp)
        want_ids[rows], want_probs[rows] = ids.cpu(), pr.cpu()
    torch.cuda.synchronize()
    ks = torch.tensor([settings[b % R][4] for b in range(busy)], dtype=torch.int32)
    assert ((ks > 0) & (want_run[:busy] >= ks)).any()  # some columns suppress the empty token
    assert torch.equal(out.cpu(), want_ids)
    assert torch.equal(probs[:busy].cpu(), want_probs)
    assert (probs[busy:] == -1).all()  # idle columns sample nothing
    assert torch.equal(run.cpu(), want_run)
    want_cur = [forced_next[b] if forced_next[b] >= 0 else int(want_ids[b]) for b in range(busy)] + [7] * idle
    assert cur.cpu().tolist() == want_cur


def test_sample_step_run_continues_resets_and_unkept_samples():
    """Argmax draws with the empty token on top: it is suppressed exactly when the run over the column's inputs reaches
    k = 3.  The run continues unless the column's request starts at this step; out_off = -1 keeps nothing; without
    forced tokens every column's next input is its sample."""
    E, k, step = EMPTY, 3, 8
    logits = torch.zeros(4, V)
    logits[:, E], logits[:, 11] = 50.0, 40.0
    settings = [(1, 32, 1, E, k, 0.0, 0.0)]
    run = torch.tensor([2, 2, 2, 1], dtype=torch.int32, device="cuda")
    cur = torch.tensor([E, E, 5, E], dtype=torch.int64, device="cuda")
    out = torch.full((4,), -9, dtype=torch.int64, device="cuda")
    # column 1 starts its request at this step; columns 0, 2, 3 continue theirs
    _sample_step(logits.cuda(), [0] * 4, [0, step, 2, 3], [0, -1, -1, -1], None, settings, run, cur, out, step)
    torch.cuda.synchronize()
    assert run.cpu().tolist() == [3, 1, 0, 2]
    assert cur.cpu().tolist() == [11, E, E, E]
    assert out.cpu().tolist() == [11, -9, -9, -9]


def test_device_rng_without_uniforms_runs_without_host_sync():
    shape, model, _ = _tiny(True)
    g = torch.Generator().manual_seed(5)
    reqs = _requests(g)
    model.generate_requests(reqs[:2], 2)  # engine creation and the parameter pack happen here, once
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = model.generate_requests(reqs, 3)
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


def test_bad_requests_raise_before_any_launch():
    shape, model, _ = _tiny(True)
    p = torch.randint(2, V, (4,))
    ok = [MT.GenRequest(p, 3), MT.GenRequest(p[:1], 2)]
    n0 = L.launch_count()
    bad = [
        ([], 2, None),
        ([MT.GenRequest(p[:0], 3)], 2, None),
        ([MT.GenRequest(p, 0)], 2, None),
        (ok, 0, None),
        ([MT.GenRequest(p, 3, technique="beam")], 2, None),
        (ok, 2, [torch.rand(3)]),
        (ok, 2, [torch.rand(3), torch.rand(3)]),
        (ok, 2, [torch.rand(3), torch.rand(2, 1)]),
    ]
    for reqs, bs, u in bad:
        with pytest.raises(ValueError):
            model.generate_requests(reqs, bs, uniforms=u)
    model.reset_length(1, 0)
    with pytest.raises(ValueError):
        model.generate_requests(ok, 2)
    assert L.launch_count() == n0
